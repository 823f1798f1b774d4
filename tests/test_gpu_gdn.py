"""Gated delta rule (torchrua_b200.delta) against an fp64 oracle on the same GPU.

The oracle is the recurrence on the zero-padded (B, T, H, K, V) state, a loop over T vectorised over the batch and
masked by length; its gradients come from autograd.  Three closed forms check the oracle itself: beta = 0, one-token
sequences written out by hand, and mutually orthogonal keys, where the rule is the SSD scan (checked against the
library's segment_ssd as well).

Inputs: k is L2-normalised, beta in (0, 1) (one case in (0, 2), where the state has negative eigenvalues but stays
stable), g <= 0 with exp(g) (1 + beta |k|^2) <= 1, so the computation on absolute values below stays bounded.

Tolerances: every output and gradient within 16 u_acc n s + c u_pay s (plus one storage ulp of |ref| for 16-bit
outputs), where s is the same computation on absolute values (|v|, |q|, |k|, |beta|, |initial|, |grad_out|, with the
delta rule's subtraction of the state's prediction turned into an addition) and n the number of terms that reach it: the
sequence's length, plus the heads of a group for grad_q / grad_k.  grad_g_r is the sum over t >= r of the in-chunk
d(cum_t), whose decay terms cancel between rows and columns: it is exactly 0 at a first token without an initial state,
but its rounding error follows the terms that cancel, so its s is the sum of s over the sequence.  u_acc is the unit
roundoff of the accumulator (2^-24, 2^-53 for fp64).  u_pay is the unit roundoff of a 16-bit PAYLOAD (2^-11, 2^-8;
0 for fp32 and fp64): the kernels round every tensor-core operand to the payload once.  The longest chain in one term
is T (rounded), Z = beta (v - gam K S_in) (which reads the rounded state copy), V' = T Z (rounded), and w V' (rounded again) in the state update; in the backward
dV', dT, X = T^T dT and dA add three more, so c = 32 covers about eight roundings with margin.
"""

import numpy as np
import pytest
import torch

import torchrua_b200 as rua

pytestmark = pytest.mark.gpu

DEV = 'cuda'
DTYPES = [torch.float32, torch.float64, torch.float16, torch.bfloat16]
ULP = {torch.float16: 2.0 ** -10, torch.bfloat16: 2.0 ** -7}
U_PAY = {torch.float16: 2.0 ** -11, torch.bfloat16: 2.0 ** -8}
C_PAY = 32
Q = 64   # chunk length of the 16-bit kernels (32 for fp32, 16 for fp64)


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


def oracle(v, lens, q, k, g, beta, h0=None, scale=None, reverse=False, magnitude=False):
    """(o (sum(lens), H, V), final (B, H, K, V)) from C rows v (rows, H, V), q, k (rows, G, K), g, beta (rows, H).
    magnitude: u = beta (v + S'^T k), the computation on absolute values (the scale s of the tolerances)."""
    H, V = v.shape[1:]
    G, K = q.shape[1:]
    scale = K ** -0.5 if scale is None else scale
    vp, valid = pad(v, lens)
    qp, _ = pad(q.repeat_interleave(H // G, dim=1), lens)
    kp, _ = pad(k.repeat_interleave(H // G, dim=1), lens)
    gp, _ = pad(g, lens)
    bp, _ = pad(beta, lens)
    B, T = valid.shape
    S = torch.zeros((B, H, K, V), dtype=v.dtype, device=v.device) if h0 is None else h0
    os_ = [None] * T
    sign = 1.0 if magnitude else -1.0
    for t in (range(T - 1, -1, -1) if reverse else range(T)):
        Sp = torch.exp(gp[:, t])[..., None, None] * S
        pred = (Sp * kp[:, t, :, :, None]).sum(-2)
        u = bp[:, t, :, None] * (vp[:, t] + sign * pred)
        Sn = Sp + kp[:, t, :, :, None] * u[:, :, None, :]
        S = torch.where(valid[:, t, None, None, None], Sn, S)
        os_[t] = scale * (S * qp[:, t, :, :, None]).sum(-2)
    o = torch.stack(os_, 1)[valid] if T else v[:0]
    return o, S


def make(lens_list, H, G, K, V, dtype, seed=0, init=False, extra_rows=0, beta_max=1.0):
    gen = torch.Generator(device=DEV).manual_seed(seed)
    lens = torch.tensor(lens_list, dtype=torch.long, device=DEV)
    rows = int(lens.sum()) + extra_rows

    def r(*s):
        return torch.randn(s, generator=gen, device=DEV, dtype=torch.float64)

    def u(*s):
        return torch.rand(s, generator=gen, device=DEV, dtype=torch.float64)

    v = r(rows, H, V).to(dtype)
    q = (r(rows, G, K) / K ** 0.25).to(dtype)
    k = torch.nn.functional.normalize(r(rows, G, K), dim=-1).to(dtype)
    beta = (beta_max * (0.05 + 0.9 * u(rows, H))).to(dtype)
    # exp(g) (1 + beta) <= 1 keeps the computation on absolute values bounded
    g = (-torch.log1p(beta.double()) - 0.3 * u(rows, H)).to(acc_of(dtype))
    h0 = (r(len(lens_list), H, K, V) / K ** 0.5).to(acc_of(dtype)) if init else None
    return lens, v, q, k, g, beta, h0


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
    """dtype: the payload's; a 16-bit result (o and the v, q, k, beta gradients) adds one storage ulp of |ref|"""
    out_ulp = ULP.get(got.dtype, 0.0)
    got, ref = got.double(), ref.double()
    u_acc = 2.0 ** -53 if dtype == torch.float64 else 2.0 ** -24
    tol = 16 * u_acc * n * s
    if dtype in U_PAY:
        tol = tol + C_PAY * U_PAY[dtype] * s + out_ulp * ref.abs() + 2.0 ** -24
    err = (got - ref).abs()
    assert bool((err <= tol).all()), (what, float(err.max()), float((err / (tol + 1e-300)).max()))


def bcast(v, like):
    return v.reshape(v.shape + (1,) * (like.dim() - v.dim()))


# ---------------------------------------------------------------------------------------------------------------------
# the oracle itself
# ---------------------------------------------------------------------------------------------------------------------
def test_oracle_beta_zero():
    """beta = 0: o = scale exp(cum) q^T initial"""
    lens, v, q, k, g, beta, h0 = make([1, 4, 0, 6], 4, 2, 3, 5, torch.float64, seed=1, init=True)
    o, fin = oracle(v, lens, q, k, g, torch.zeros_like(beta), h0)
    seq = torch.repeat_interleave(torch.arange(4, device=DEV), lens)
    off = torch.cumsum(lens, 0) - lens
    cum = torch.cat([torch.cumsum(g[o_:o_ + n], 0) for o_, n in zip(off.tolist(), lens.tolist())])
    ref = 3 ** -0.5 * torch.exp(cum)[..., None] * torch.einsum('rhk,rhkv->rhv', q.repeat_interleave(2, 1), h0[seq])
    assert float((o - ref).abs().max()) <= 1e-12
    assert torch.equal(fin[2], h0[2])


def test_oracle_one_token():
    """one-token sequences written out by hand"""
    lens, v, q, k, g, beta, h0 = make([1, 1, 1], 2, 1, 4, 3, torch.float64, seed=2, init=True)
    o, fin = oracle(v, lens, q, k, g, beta, h0, scale=0.7)
    for i in range(3):
        for h in range(2):
            Sp = torch.exp(g[i, h]) * h0[i, h]
            u = beta[i, h] * (v[i, h] - Sp.T @ k[i, 0])
            S = Sp + torch.outer(k[i, 0], u)
            assert float((fin[i, h] - S).abs().max()) <= 1e-13
            assert float((o[i, h] - 0.7 * S.T @ q[i, 0]).abs().max()) <= 1e-13


@pytest.mark.parametrize('dtype', [torch.float32, torch.float64], ids=str)
def test_orthogonal_keys_match_ssd(dtype):
    """k_t = e_t (T <= K), no initial: the projection term vanishes and the rule is the SSD scan with delta = -g,
    A = -1, x = beta v / delta, B = k, C = scale q and the state transposed"""
    H, G, K, V = 4, 2, 32, 24
    lens_list = [0, 1, 17, 32, 5]
    lens, v, q, _, g, beta, _ = make(lens_list, H, G, K, V, dtype, seed=3)
    k = torch.cat([torch.eye(K, dtype=dtype, device=DEV)[:n] for n in lens_list])[:, None].expand(-1, G, K).contiguous()
    scale = 0.5
    o, fin = rua.segment_gated_delta_rule(v, lens, q, k, g, beta, scale=scale, return_final_state=True)
    delta = (-g).to(dtype)
    x = beta[..., None] * v / delta[..., None]
    y, hf = rua.segment_ssd(x, lens, delta, -torch.ones(H, dtype=acc_of(dtype), device=DEV), k, scale * q,
                            return_final_state=True)
    o_ref, f_ref = oracle(d64(v), lens, d64(q), d64(k), d64(g), d64(beta), scale=scale)
    tol = 1e-5 if dtype == torch.float32 else 1e-12
    torch.testing.assert_close(o.double(), o_ref, atol=tol, rtol=tol)
    torch.testing.assert_close(fin.double(), f_ref, atol=tol, rtol=tol)
    torch.testing.assert_close(y.double(), o_ref, atol=tol, rtol=tol)
    torch.testing.assert_close(hf.transpose(-1, -2).double(), f_ref, atol=tol, rtol=tol)


# ---------------------------------------------------------------------------------------------------------------------
# forward + backward through a layout against the oracle
# ---------------------------------------------------------------------------------------------------------------------
def run_case(kind, lens, v, q, k, g, beta, h0, reverse, dtype, seed=0, scale=None):
    """checks o, final and the six gradients against the oracle; returns (out, fin, leaves)"""
    zv, back = as_layout(kind, lens, v)
    parts = [as_layout(kind, lens, t)[0].data for t in (q, k, g, beta)]
    leaves = [zv.data.detach().requires_grad_(True)] + [t.detach().requires_grad_(True) for t in parts] + \
        [None if h0 is None else h0.detach().requires_grad_(True)]
    out, fin = zv._replace(data=leaves[0]).gated_delta_rule(*leaves[1:5], scale=scale, initial=leaves[5],
                                                            reverse=reverse, return_final_state=True)
    assert type(out) is type(zv) and out.data.dtype == dtype and fin.dtype == acc_of(dtype) and not fin.requires_grad
    go = torch.randn(out.data.shape, generator=torch.Generator(device=DEV).manual_seed(seed + 1), device=DEV,
                     dtype=torch.float64).to(dtype)
    out.data.backward(go)
    refs = [None if t is None else t.requires_grad_(True) for t in map(d64, (v, q, k, g, beta, h0))]
    o_ref, f_ref = oracle(*refs[:1], lens, *refs[1:5], refs[5], scale, reverse)
    gc = back(go).double().reshape(o_ref.shape)
    (o_ref * gc).sum().backward()
    mags = [None if t is None else t.detach().abs().requires_grad_(True) for t in refs]
    mags[3] = refs[3].detach().requires_grad_(True)
    o_s, f_s = oracle(*mags[:1], lens, *mags[1:5], mags[5], scale, reverse, magnitude=True)
    (o_s * gc.abs()).sum().backward()
    H, G = v.shape[1], q.shape[1]
    per_row = torch.repeat_interleave(lens.double(), lens)
    within(back(out.data).reshape(o_ref.shape), o_ref, o_s.detach(), bcast(per_row, o_ref), dtype, 'o')
    within(fin, f_ref, f_s.detach(), bcast(lens.double(), f_ref), dtype, 'final')
    nterms = [per_row, per_row + H // G, per_row + H // G, per_row, per_row, lens.double()]
    for j, name in enumerate(['v', 'q', 'k', 'g', 'beta', 'initial']):
        if leaves[j] is None:
            continue
        got = leaves[j].grad
        if j < 5:
            got = back(got).reshape(refs[j].shape)
        s = mags[j].grad.abs() if mags[j].grad is not None else torch.zeros_like(refs[j])
        if name == 'g':   # a difference of in-chunk sums (rows minus columns): its error follows the whole sequence
            seq = torch.repeat_interleave(torch.arange(lens.numel(), device=DEV), lens)
            s = torch.zeros((lens.numel(),) + s.shape[1:], dtype=s.dtype, device=DEV).index_add_(0, seq, s)[seq]
        within(got.reshape(refs[j].shape), refs[j].grad, s, bcast(nterms[j], refs[j]), dtype, 'grad_' + name)
    return out, fin, leaves


GRID_LENS = [0, 1, 3, 7, 2, 0, 13, 5, 1, 9, 33, 70]
SHAPES = [(1, 1, 1, 1), (3, 1, 7, 5), (2, 2, 128, 128), (8, 4, 128, 64), (4, 2, 64, 256)]


@pytest.mark.parametrize('reverse', [False, True], ids=['fwd', 'rev'])
@pytest.mark.parametrize('init', [False, True], ids=['noh0', 'h0'])
@pytest.mark.parametrize('shape', SHAPES, ids=lambda s: 'H%dG%dK%dV%d' % s)
@pytest.mark.parametrize('kind', ['C', 'L', 'P', 'R'])
@pytest.mark.parametrize('dtype', DTYPES, ids=str)
def test_grid(dtype, kind, shape, init, reverse):
    H, G, K, V = shape
    lens, v, q, k, g, beta, h0 = make(GRID_LENS, H, G, K, V, dtype, seed=H * 7 + K, init=init)
    out, fin, leaves = run_case(kind, lens, v, q, k, g, beta, h0, reverse, dtype)
    if kind in ('L', 'R'):   # padding rows: o copies v, grad_v = grad_out, the other gradients 0
        mask = rua.C(data=torch.ones(int(lens.sum()), device=DEV), token_sizes=lens)
        mz, _ = as_layout(kind, lens, mask.data)
        pad_rows = mz.data == 0
        zv, _ = as_layout(kind, lens, v)
        assert torch.equal(out.data[pad_rows], zv.data[pad_rows])
        for j in (1, 2, 3, 4):
            assert bool((leaves[j].grad[pad_rows] == 0).all())


@pytest.mark.parametrize('kind, init, reverse', [('C', True, False), ('L', False, True), ('P', False, False),
                                                 ('R', True, True)], ids=['C-h0-fwd', 'L-noh0-rev', 'P-noh0-fwd',
                                                                          'R-h0-rev'])
@pytest.mark.parametrize('dtype', DTYPES, ids=str)
def test_qwen_next_heads(dtype, kind, init, reverse):
    """H = 32 value heads over G = 16 key groups, K = V = 128, at a small batch: every layout, with and without an
    initial state, in both directions"""
    lens, v, q, k, g, beta, h0 = make([5, 0, 40, 1, 70], 32, 16, 128, 128, dtype, seed=20, init=init)
    run_case(kind, lens, v, q, k, g, beta, h0, reverse, dtype)


@pytest.mark.parametrize('reverse', [False, True], ids=['fwd', 'rev'])
@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16], ids=str)
def test_slow_decay(dtype, reverse):
    """g in (-0.05, 0), the gates of trained models, over a few hundred tokens: the state carries information across
    many chunks, so errors carried from chunk to chunk are exercised.

    Here the computation on absolute values grows like 2^t and gives no bound, so the check is normwise per tensor:
    ||got - ref|| <= (16 u_acc n + 8 u_pay (1 + ceil(n / Q))) ||ref||, n the longest length.  Every map that carries the
    state or its adjoint from one chunk to the next has norm <= 1 (exp(g) <= 1, and I - beta k k^T with beta in (0, 1]
    and |k| = 1), so the roundings of each chunk are carried without growth and add up over the chunks; within a chunk
    a term passes through about eight roundings to the payload (the chain in the module docstring, and the rounding of
    the stored result), one payload unit each."""
    lens_list = [300, 257, 1, 64, 130]
    lens, v, q, k, _, beta, h0 = make(lens_list, 4, 2, 64, 64, dtype, seed=23, init=True)
    g = -0.05 * torch.rand(beta.shape, generator=torch.Generator(device=DEV).manual_seed(24), device=DEV,
                           dtype=torch.float64).to(acc_of(dtype))
    leaves = [t.detach().requires_grad_(True) for t in (v, q, k, g, beta, h0)]
    o, fin = rua.segment_gated_delta_rule(leaves[0], lens, *leaves[1:5], initial=leaves[5], reverse=reverse,
                                          return_final_state=True)
    go = torch.randn(o.shape, generator=torch.Generator(device=DEV).manual_seed(25), device=DEV,
                     dtype=torch.float64).to(dtype)
    o.backward(go)
    refs = [t.requires_grad_(True) for t in map(d64, (v, q, k, g, beta, h0))]
    o_ref, f_ref = oracle(refs[0], lens, *refs[1:5], refs[5], None, reverse)
    (o_ref * go.double()).sum().backward()
    n = max(lens_list)
    u_acc, u_pay = 2.0 ** -24, U_PAY.get(dtype, 0.0)
    rel = 16 * u_acc * n + 8 * u_pay * (1 + -(-n // Q))
    pairs = [('o', o, o_ref), ('final', fin, f_ref)] + \
        [('grad_' + name, t.grad, r.grad) for name, t, r in zip(['v', 'q', 'k', 'g', 'beta', 'initial'], leaves, refs)]
    for what, got, ref in pairs:
        err, size = float((got.detach().double() - ref.detach()).norm()), float(ref.detach().norm())
        assert err <= rel * size, (what, err / size, rel)


@pytest.mark.parametrize('reverse', [False, True])
@pytest.mark.parametrize('dtype', DTYPES, ids=str)
def test_chunk_boundaries(dtype, reverse):
    lens_list = [0, 1, Q - 1, Q, Q + 1, 2 * Q, 2 * Q + 1, 17, 15, 16, 31, 32, 33]
    lens, v, q, k, g, beta, h0 = make(lens_list, 4, 2, 40, 72, dtype, seed=3, init=True)
    for kind in ('C', 'P'):
        run_case(kind, lens, v, q, k, g, beta, h0, reverse, dtype)


@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16], ids=str)
def test_negative_eigenvalues(dtype):
    """beta in (0, 2): I - beta k k^T has a negative eigenvalue, the state stays bounded"""
    lens, v, q, k, g, beta, h0 = make([1, 70, 129, 3], 4, 2, 32, 48, dtype, seed=21, init=True, beta_max=2.0)
    run_case('C', lens, v, q, k, g, beta, h0, False, dtype, scale=0.3)


@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16], ids=str)
def test_long_and_zipf_sequences(dtype):
    """a 4096-token sequence next to short ones, and Zipf lengths (cfg3-like, capped at 4096) at a small H"""
    rng = np.random.default_rng(5)
    zipf = np.minimum(rng.zipf(1.3, size=40), 4096).tolist()
    lens, v, q, k, g, beta, h0 = make([4096, 1, 0, 300] + zipf, 2, 1, 32, 16, dtype, seed=4, init=True)
    run_case('C', lens, v, q, k, g, beta, h0, False, dtype)


def test_many_short_sequences():
    """32768 short sequences: the backward grid is capped and every CTA walks many units"""
    rng = np.random.default_rng(6)
    lens_list = rng.integers(0, 6, size=32768).tolist()
    lens, v, q, k, g, beta, h0 = make(lens_list, 2, 1, 16, 8, torch.float32, seed=6, init=True)
    run_case('C', lens, v, q, k, g, beta, h0, True, torch.float32)


def test_rows_past_the_tokens():
    """C storage longer than sum(sizes): o copies v there, grad_v passes grad_out, the other gradients are 0"""
    lens, v, q, k, g, beta, _ = make([3, 5, 0, 2], 4, 2, 8, 16, torch.float32, seed=6, extra_rows=7)
    leaves = [t.detach().requires_grad_(True) for t in (v, q, k, g, beta)]
    o = rua.segment_gated_delta_rule(leaves[0], lens, *leaves[1:])
    go = torch.randn_like(o)
    o.backward(go)
    n = int(lens.sum())
    assert torch.equal(o[n:], v[n:]) and torch.equal(leaves[0].grad[n:], go[n:])
    for j in (1, 2, 3, 4):
        assert bool((leaves[j].grad[n:] == 0).all())
    o0 = rua.segment_gated_delta_rule(v[:n], lens, q[:n], k[:n], g[:n], beta[:n])
    assert torch.equal(o[:n], o0)


# ---------------------------------------------------------------------------------------------------------------------
# identities
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('dtype', [torch.float32, torch.float64], ids=str)
def test_overwrite_property(dtype):
    """g = 0, beta = 1, unit k: the state stores v_last under k_last exactly, final^T k_last = v_last"""
    lens, v, q, k, g, beta, h0 = make([1, 9, 70, 130], 4, 2, 64, 32, dtype, seed=22, init=True)
    _, fin = rua.segment_gated_delta_rule(v, lens, q, k, torch.zeros_like(g), torch.ones_like(beta), initial=h0,
                                          return_final_state=True)
    last = torch.cumsum(lens, 0) - 1
    got = torch.einsum('bhkv,bhk->bhv', fin, k[last].repeat_interleave(2, 1).to(fin.dtype))
    tol = 1e-4 if dtype == torch.float32 else 1e-12
    torch.testing.assert_close(got, v[last].to(fin.dtype), atol=tol, rtol=tol)


@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16], ids=str)
def test_streaming(dtype):
    """part one's final fed as part two's initial equals the whole sequence"""
    lens, v, q, k, g, beta, h0 = make([150], 4, 2, 64, 64, dtype, seed=9, init=True)
    o, f = rua.segment_gated_delta_rule(v, lens, q, k, g, beta, initial=h0, return_final_state=True)
    cut = 70
    one, two = torch.tensor([cut], device=DEV), torch.tensor([150 - cut], device=DEV)
    o1, f1 = rua.segment_gated_delta_rule(v[:cut], one, q[:cut], k[:cut], g[:cut], beta[:cut], initial=h0,
                                          return_final_state=True)
    o2, f2 = rua.segment_gated_delta_rule(v[cut:], two, q[cut:], k[cut:], g[cut:], beta[cut:], initial=f1,
                                          return_final_state=True)
    tol = 2e-5 if dtype == torch.float32 else 3e-2
    torch.testing.assert_close(torch.cat([o1, o2]).float(), o.float(), atol=tol, rtol=tol)
    torch.testing.assert_close(f2, f, atol=tol, rtol=tol)


# ---------------------------------------------------------------------------------------------------------------------
# determinism: no leakage, bit-identical layouts and reruns
# ---------------------------------------------------------------------------------------------------------------------
def grads_of(kind, lens, v, q, k, g, beta, h0, go, reverse=False):
    zv, back = as_layout(kind, lens, v)
    parts = [as_layout(kind, lens, t)[0].data for t in (q, k, g, beta)]
    leaves = [zv.data.detach().requires_grad_(True)] + [t.detach().requires_grad_(True) for t in parts] + \
        [h0.detach().requires_grad_(True)]
    out, fin = zv._replace(data=leaves[0]).gated_delta_rule(*leaves[1:5], initial=leaves[5], reverse=reverse,
                                                            return_final_state=True)
    zg, _ = as_layout(kind, lens, go)
    out.data.backward(zg.data)
    res = [back(out.data), fin] + [back(t.grad) if j < 5 else t.grad for j, t in enumerate(leaves)]
    return [r.detach().clone() for r in res]


@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16], ids=str)
def test_bit_identical_layouts_and_reruns(dtype):
    lens, v, q, k, g, beta, h0 = make([70, 0, 5, 130, 1, 64], 4, 2, 64, 96, dtype, seed=10, init=True)
    go = torch.randn(v.shape, device=DEV, dtype=torch.float64).to(dtype)
    for reverse in (False, True):
        base = grads_of('C', lens, v, q, k, g, beta, h0, go, reverse)
        assert all(torch.equal(u, w) for u, w in zip(base, grads_of('C', lens, v, q, k, g, beta, h0, go, reverse)))
        for kind in ('L', 'P', 'R'):
            other = grads_of(kind, lens, v, q, k, g, beta, h0, go, reverse)
            for j, (u, w) in enumerate(zip(base, other)):
                assert torch.equal(u, w), (kind, reverse, j)


def test_no_leakage():
    """perturbing one sequence leaves every other sequence's outputs and gradients bit-identical"""
    lens_list = [70, 3, 0, 129]
    lens, v, q, k, g, beta, h0 = make(lens_list, 4, 2, 32, 32, torch.bfloat16, seed=11, init=True)
    go = torch.randn(v.shape, device=DEV, dtype=torch.float64).to(torch.bfloat16)
    base = grads_of('C', lens, v, q, k, g, beta, h0, go)
    off = [0] + np.cumsum(lens_list).tolist()
    r1 = slice(off[1], off[2])
    v2, q2, g2 = v.clone(), q.clone(), g.clone()
    v2[r1] += 1
    q2[r1] *= -1
    g2[r1] -= 0.1
    h2 = h0.clone()
    h2[1] += 1
    pert = grads_of('C', lens, v2, q2, k, g2, beta, h2, go)
    keep = torch.ones(v.shape[0], dtype=torch.bool, device=DEV)
    keep[r1] = False
    for j, (u, w) in enumerate(zip(base, pert)):
        if j in (1, 7):   # final, grad_initial: (B, H, K, V)
            idx = [0, 2, 3]
            assert torch.equal(u[idx], w[idx]), j
        else:
            assert torch.equal(u[keep], w[keep]), j


# ---------------------------------------------------------------------------------------------------------------------
# autograd plumbing
# ---------------------------------------------------------------------------------------------------------------------
def test_gradcheck_and_double_backward():
    lens, v, q, k, g, beta, h0 = make([3, 0, 2, 19], 2, 1, 3, 2, torch.float64, seed=12, init=True)
    args = [t.detach().requires_grad_(True) for t in (v, q, k, g, beta, h0)]

    def f(*a):
        o, fin = rua.segment_gated_delta_rule(a[0], lens, *a[1:5], initial=a[5], return_final_state=True)
        return o
    assert torch.autograd.gradcheck(f, args, eps=1e-6, atol=1e-7)
    o = f(*args)
    (gv,) = torch.autograd.grad(o.sum(), args[0], create_graph=True)
    with pytest.raises(RuntimeError):
        gv.sum().backward()


def test_partial_gradients_and_no_grad():
    """an unwanted gradient is not computed; without autograd the forward gives the same bits"""
    lens, v, q, k, g, beta, h0 = make([5, 70], 4, 2, 8, 16, torch.float32, seed=13, init=True)
    with torch.no_grad():
        o0 = rua.segment_gated_delta_rule(v, lens, q, k, g, beta, initial=h0)
    vr = v.detach().requires_grad_(True)
    o = rua.segment_gated_delta_rule(vr, lens, q, k, g, beta, initial=h0)
    assert torch.equal(o0, o.detach())
    o.sum().backward()
    assert vr.grad is not None
    full = grads_of('C', lens, v, q, k, g, beta, h0, torch.ones_like(v))
    assert torch.equal(vr.grad, full[2])
    from torchrua_b200 import _native
    from torchrua_b200._lib import CAT
    rg = _native.ragged_from_lengths(lens, want_pack=True)
    side = _native.SideSpec(CAT, rows=v.shape[0])
    only_g = _native._gdn_backward_raw(torch.ones_like(v), v, q, k, g, beta, h0, 8 ** -0.5, rg, side, False,
                                       (False, False, False, True, False, False))
    assert [t is None for t in only_g] == [True, True, True, False, True, True]
    assert torch.equal(only_g[3], full[5])


def test_sequence_longer_than_tp_gets_nan_gradients():
    """the backward's scratch is sized by ragged->Tp: a sequence longer than it gets NaN in every gradient it reaches,
    and the other sequences keep their bits"""
    import copy
    from torchrua_b200 import _native
    from torchrua_b200._lib import CAT
    lens, v, q, k, g, beta, h0 = make([70, 5, 130, 0, 20], 4, 2, 8, 16, torch.float32, seed=14, init=True)
    go = torch.randn_like(v)
    rg = _native.ragged_from_lengths(lens, want_pack=True)
    side = _native.SideSpec(CAT, rows=v.shape[0])
    want = (True,) * 6
    full = _native._gdn_backward_raw(go, v, q, k, g, beta, h0, 0.5, rg, side, False, want)
    short = copy.copy(rg)
    short.Tp = 100
    cut = _native._gdn_backward_raw(go, v, q, k, g, beta, h0, 0.5, short, side, False, want)
    o = torch.cumsum(lens, 0) - lens
    bad = slice(int(o[2]), int(o[2]) + 130)
    keep = torch.ones(v.shape[0], dtype=torch.bool, device=DEV)
    keep[bad] = False
    for j in range(5):
        assert bool(cut[j][bad].isnan().all())
        assert torch.equal(cut[j][keep], full[j][keep])
    assert bool(cut[5][2].isnan().all()) and torch.equal(cut[5][[0, 1, 3, 4]], full[5][[0, 1, 3, 4]])
