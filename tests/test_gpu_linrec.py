"""Per-sequence gated linear recurrence (segment_linear_recurrence and the layout methods) against the recurrence in fp64,
looped over T on the zero-padded (B, T, *feat) batch on the same GPU, and its autograd for the gradients."""
import numpy as np
import pytest
import torch

import torchrua_b200 as rua

pytestmark = pytest.mark.gpu

DEV = torch.device('cuda')
DTYPES = [torch.float32, torch.float64, torch.float16, torch.bfloat16]
LAYOUTS = ['C', 'L', 'P', 'R']
FEATS = [(), (1,), (7,), (1024,), (4, 8)]


def _inputs(lens, feat, dtype, seed=0, gate='uniform', initial=False):
    g = torch.Generator().manual_seed(seed)
    shape = (int(sum(lens)),) + tuple(feat)
    x = torch.randn(shape, generator=g, dtype=torch.float64)
    if gate == 'uniform':
        a = torch.rand(shape, generator=g, dtype=torch.float64)
    elif gate == 'signed':
        a = torch.rand(shape, generator=g, dtype=torch.float64) * 2.2 - 1.1
    else:
        a = torch.full(shape, float(gate), dtype=torch.float64)
    h0 = torch.randn((len(lens),) + tuple(feat), generator=g, dtype=torch.float64) if initial else None
    to = lambda t: None if t is None else t.to(dtype).to(DEV)   # noqa: E731
    return to(x), to(a), to(h0), torch.tensor(lens, dtype=torch.long, device=DEV)


def _rev_rows(lens):
    """C row of token (i, len-1-t) for every C row (i, t), and t"""
    lens = torch.as_tensor(lens, dtype=torch.long)
    off = torch.cumsum(lens, 0) - lens
    seg = torch.repeat_interleave(torch.arange(lens.numel()), lens)
    t = torch.arange(int(lens.sum())) - off[seg]
    return (off[seg] + lens[seg] - 1 - t).to(DEV), t.to(DEV), seg.to(DEV)


def oracle(x, a, h0, lens, reverse):
    """the recurrence in fp64 (differentiable), looped over T, vectorised over B and the features; C order in and out"""
    rrows, t, seg = _rev_rows(lens)
    x, a = x.double(), a.double()
    if reverse:
        x, a = x[rrows], a[rrows]
    B, T, feat = len(lens), max(list(lens) + [1]), tuple(x.shape[1:])
    px = torch.zeros((B, T) + feat, dtype=torch.float64, device=DEV).index_put((seg, t), x)
    pa = torch.zeros((B, T) + feat, dtype=torch.float64, device=DEV).index_put((seg, t), a)
    h = torch.zeros((B,) + feat, dtype=torch.float64, device=DEV) if h0 is None else h0.double()
    outs = []
    for k in range(T):
        h = pa[:, k] * h + px[:, k]
        outs.append(h)
    y = torch.stack(outs, 1)[seg, t]
    return y[rrows] if reverse else y


def check_close(got, ref, x, a, h0, lens, reverse, what=''):
    scale = oracle(x.abs(), a.abs(), None if h0 is None else h0.abs(), lens, reverse)
    if x.dtype == torch.float64:
        tol = 1e-12
    elif x.dtype == torch.float32:
        tol = 1e-5
    else:
        tol = 1e-2
        ref = ref.to(x.dtype).double()   # the fp64 result rounded once
    err = (got.double() - ref).abs()
    bad = ~(err <= tol * ref.abs() + tol * scale)
    assert not bad.any(), f'{what} {x.dtype}: max err {err[bad].max().item()} at {bad.nonzero()[:4].tolist()}'


def make_layout(kind, t, lens):
    c = rua.C(data=t, token_sizes=lens)
    if kind == 'C':
        return c
    if kind == 'P':
        return c.pack()
    return c.left(0) if kind == 'L' else c.right(0)


def run_layout(kind, x, a, h0, lens, reverse):
    z, za = make_layout(kind, x, lens), make_layout(kind, a, lens)
    out = z.linear_recurrence(za.data, h0, reverse=reverse)
    assert type(out) is type(z)
    return out.cat().data


@pytest.mark.parametrize('initial', [False, True])
@pytest.mark.parametrize('reverse', [False, True])
@pytest.mark.parametrize('kind', LAYOUTS)
@pytest.mark.parametrize('dtype', DTYPES)
def test_forward_parity(dtype, kind, reverse, initial):
    for k, feat in enumerate(FEATS):
        lens = [[3, 0, 5, 1, 7, 2, 0], [1], [4, 9, 0, 6], [40, 3, 17, 0, 2], [5, 0, 3, 8]][k]
        x, a, h0, ls = _inputs(lens, feat, dtype, seed=k, initial=initial)
        ref = oracle(x, a, h0, lens, reverse)
        check_close(run_layout(kind, x, a, h0, ls, reverse), ref, x, a, h0, lens, reverse, f'{kind} {feat}')
        free = rua.segment_linear_recurrence(x, ls, a, h0, reverse=reverse)
        check_close(free, ref, x, a, h0, lens, reverse, f'free {feat}')


@pytest.mark.parametrize('dtype', DTYPES)
def test_gate_cases(dtype):
    lens = [6, 0, 11, 1, 300]
    for reverse in (False, True):
        for kind in LAYOUTS:
            x, a, h0, ls = _inputs(lens, (32,), dtype, seed=1, gate='signed', initial=True)
            check_close(run_layout(kind, x, a, h0, ls, reverse), oracle(x, a, h0, lens, reverse), x, a, h0, lens, reverse,
                        'signed')
            # a = 0 returns x bit-exactly, whatever the initial state
            x, a, h0, ls = _inputs(lens, (32,), dtype, seed=2, gate=0.0, initial=True)
            assert torch.equal(run_layout(kind, x, a, h0, ls, reverse), x)
        # a = 1 is cumsum
        x, a, _, ls = _inputs(lens, (32,), dtype, seed=3, gate=1.0)
        got = rua.segment_linear_recurrence(x, ls, a, reverse=reverse)
        ref = oracle(x, a, None, lens, reverse)
        check_close(got, ref, x, a, None, lens, reverse, 'a=1')
        check_close(rua.segment_cumsum(x, ls, reverse=reverse), ref, x, a, None, lens, reverse, 'cumsum')


def _grads(fn, leaves, g):
    leaves = [t.clone().requires_grad_(True) for t in leaves]
    y = fn(*leaves)
    return y.detach(), torch.autograd.grad(y, leaves, g)


@pytest.mark.parametrize('dtype', [torch.float32, torch.float64, torch.bfloat16])
@pytest.mark.parametrize('kind', LAYOUTS)
def test_gradients_against_oracle(kind, dtype):
    lens = [6, 0, 11, 1, 300, 2]
    x, a, h0, ls = _inputs(lens, (16,), dtype, seed=4, gate='signed', initial=True)
    for reverse in (False, True):
        g = torch.randn_like(x)

        def ours(xx, aa, hh):
            z, za = make_layout(kind, xx, ls), make_layout(kind, aa, ls)
            return z.linear_recurrence(za.data, hh, reverse=reverse).cat().data

        _, got = _grads(ours, (x, a, h0), g)
        _, want = _grads(lambda xx, aa, hh: oracle(xx, aa, hh, lens, reverse), (x.double(), a.double(), h0.double()),
                         g.double())
        tol = {torch.float64: 1e-10, torch.float32: 1e-4}.get(dtype, 3e-2)
        for name, u, v in zip(('x', 'gate', 'initial'), got, want):
            torch.testing.assert_close(u.double(), v, rtol=tol, atol=tol * (1 + v.abs().max().item()), msg=name)


@pytest.mark.parametrize('kind', LAYOUTS)
def test_gradcheck_fp64(kind):
    lens = [3, 0, 4, 1]
    x, a, h0, ls = _inputs(lens, (3,), torch.float64, seed=5, gate='signed', initial=True)
    for reverse in (False, True):
        def f(xx, aa, hh):
            z, za = make_layout(kind, xx, ls), make_layout(kind, aa, ls)
            return z.linear_recurrence(za.data, hh, reverse=reverse).cat().data
        assert torch.autograd.gradcheck(f, tuple(t.clone().requires_grad_(True) for t in (x, a, h0)))


def test_frozen_inputs_and_double_backward():
    lens = [4, 0, 7]
    x, a, h0, ls = _inputs(lens, (5,), torch.float64, seed=6, initial=True)
    # frozen gate: no gate gradient, and y is not kept for it
    xx, hh = x.clone().requires_grad_(True), h0.clone().requires_grad_(True)
    y = rua.segment_linear_recurrence(xx, ls, a, hh)
    assert y.grad_fn.saved_tensors[2] is None
    gx, gh = torch.autograd.grad(y.sum(), (xx, hh))
    _, want = _grads(lambda u, v: oracle(u, a, v, lens, False), (x, h0), torch.ones_like(x))
    torch.testing.assert_close(gx, want[0])
    torch.testing.assert_close(gh, want[1])
    # frozen x: the gate gradient alone, y kept
    aa = a.clone().requires_grad_(True)
    y = rua.segment_linear_recurrence(x, ls, aa, h0)
    assert y.grad_fn.saved_tensors[2] is not None
    (ga,) = torch.autograd.grad(y.sum(), aa)
    _, want = _grads(lambda v: oracle(x, v, h0, lens, False), (a,), torch.ones_like(x))
    torch.testing.assert_close(ga, want[0])
    # once-differentiable
    xx = x.clone().requires_grad_(True)
    y = rua.segment_linear_recurrence(xx, ls, a)
    (g,) = torch.autograd.grad((y ** 2).sum(), xx, create_graph=True)
    with pytest.raises(RuntimeError):
        torch.autograd.grad(g.sum(), xx)


@pytest.mark.parametrize('reverse', [False, True])
@pytest.mark.parametrize('dtype', [torch.float32, torch.float64])
def test_streaming_across_chunks(dtype, reverse):
    rng = np.random.default_rng(7)
    lens = rng.integers(2, 200, 64).tolist()
    cut = [int(rng.integers(1, n)) for n in lens]
    x, a, _, ls = _inputs(lens, (24,), dtype, seed=7)
    off = np.concatenate([[0], np.cumsum(lens)])
    first = torch.tensor(np.concatenate([np.arange(o, o + k) for o, k in zip(off[:-1], cut)]), device=DEV)
    second = torch.tensor(np.concatenate([np.arange(o + k, o + n) for o, k, n in zip(off[:-1], cut, lens)]), device=DEV)
    l1 = torch.tensor(cut, device=DEV)
    l2 = ls - l1
    if reverse:   # the later part runs first and hands its state to the earlier one
        first, second, l1, l2 = second, first, l2, l1
    whole = rua.segment_linear_recurrence(x, ls, a, reverse=reverse)
    y1 = rua.C(data=rua.segment_linear_recurrence(x[first], l1, a[first], reverse=reverse), token_sizes=l1)
    state = y1.head(1).data if reverse else y1.last()
    h = state.clone().requires_grad_(True)
    y2 = rua.segment_linear_recurrence(x[second], l2, a[second], h, reverse=reverse)
    tol = 1e-12 if dtype == torch.float64 else 1e-5
    torch.testing.assert_close(y1.data, whole[first], rtol=tol, atol=tol)
    torch.testing.assert_close(y2.detach(), whole[second], rtol=tol, atol=tol * 10)
    # grad_initial of the second call = the whole-sequence gradient at the last row of the first part
    g = torch.randn_like(y2)
    (gh,) = torch.autograd.grad(y2, h, g)
    xx = x.clone().requires_grad_(True)
    gw = torch.zeros_like(x)
    gw[second] = g
    (gx,) = torch.autograd.grad(rua.segment_linear_recurrence(xx, ls, a, reverse=reverse), xx, gw)
    edge = torch.tensor([o + k - 1 for o, k in zip(off[:-1], cut)], device=DEV) if not reverse else \
        torch.tensor([o + k for o, k in zip(off[:-1], cut)], device=DEV)
    torch.testing.assert_close(gh, gx[edge], rtol=tol * 10, atol=tol * 10)


@pytest.mark.parametrize('kind', LAYOUTS)
def test_long_sequences_across_many_chunks(kind):
    lens = [1, 20000, 3, 5000]
    for dtype in (torch.float32, torch.float64):
        x, a, h0, ls = _inputs(lens, (4,), dtype, seed=8, gate='signed', initial=True)
        for reverse in (False, True):
            check_close(run_layout(kind, x, a, h0, ls, reverse), oracle(x, a, h0, lens, reverse), x, a, h0, lens, reverse,
                        f'long {kind}')


def test_many_narrow_sequences():
    rng = np.random.default_rng(9)
    lens = rng.integers(1, 64, 32768)
    lens[::97] = 0
    lens[5000] = 1500
    lens = lens.tolist() + [0, 0, 0]
    x, a, h0, ls = _inputs(lens, (1,), torch.float32, seed=9, initial=True)
    for reverse in (False, True):
        got = rua.segment_linear_recurrence(x, ls, a, h0, reverse=reverse)
        check_close(got, oracle(x, a, h0, lens, reverse), x, a, h0, lens, reverse, 'narrow')


def test_empty_sequences_with_initial():
    lens = [0, 3, 0, 0, 2, 0]
    x, a, h0, ls = _inputs(lens, (8,), torch.float32, seed=10, initial=True)
    xx, aa, hh = (t.clone().requires_grad_(True) for t in (x, a, h0))
    y = rua.segment_linear_recurrence(xx, ls, aa, hh)
    check_close(y.detach(), oracle(x, a, h0, lens, False), x, a, h0, lens, False, 'empty')
    gx, ga, gh = torch.autograd.grad(y, (xx, aa, hh), torch.randn_like(y))
    assert (gh[[0, 2, 3, 5]] == 0).all() and (gh[[1, 4]] != 0).any()
    # no token at all: nothing to compute, grad_initial is 0
    e = torch.zeros(0, 8, device=DEV, requires_grad=True)
    he = torch.randn(2, 8, device=DEV, requires_grad=True)
    ye = rua.segment_linear_recurrence(e, torch.zeros(2, dtype=torch.long, device=DEV), e.detach(), he)
    assert ye.shape == (0, 8)
    (ghe,) = torch.autograd.grad(ye.sum() + 0 * he.sum(), he)
    assert (ghe == 0).all()


@pytest.mark.parametrize('kind', ['L', 'R'])
def test_padding_rows(kind):
    lens = [3, 0, 5, 2]
    x, a, h0, ls = _inputs(lens, (8,), torch.float32, seed=11, initial=True)
    z, za = make_layout(kind, x, ls), make_layout(kind, a, ls)
    extra = 3
    b = z.data.shape[0]
    pad = torch.full((b, extra, 8), 7.0, device=DEV)
    wide = (lambda t: torch.cat([t, pad], 1)) if kind == 'L' else (lambda t: torch.cat([pad, t], 1))
    data, gate = wide(z.data).requires_grad_(True), wide(za.data).requires_grad_(True)
    y = z._replace(data=data).linear_recurrence(gate, h0)
    tok = make_layout(kind, torch.ones(len(x), 1, device=DEV), ls).data[..., 0] > 0
    none = torch.zeros(b, extra, dtype=torch.bool, device=DEV)
    tok = torch.cat([tok, none], 1) if kind == 'L' else torch.cat([none, tok], 1)
    assert torch.equal(y.data[~tok].detach(), data.detach()[~tok])
    # the token rows in row-major order are the C order of the tokens
    check_close(y.data[tok].detach(), oracle(x, a, h0, lens, False), x, a, h0, lens, False, 'padded')
    g = torch.randn_like(y.data)
    gx, ga = torch.autograd.grad(y.data, (data, gate), g)
    assert torch.equal(gx[~tok], g[~tok])
    assert (ga[~tok] == 0).all()


def cfg3_lengths(B=16384, seed=0):
    rng = np.random.default_rng(seed)
    return np.minimum(rng.zipf(1.5, B), 4096).tolist()


def test_cfg3_lengths_and_determinism():
    lens = cfg3_lengths()
    x, a, h0, ls = _inputs(lens, (8,), torch.float32, seed=12, initial=True)
    for reverse in (False, True):
        got = rua.segment_linear_recurrence(x, ls, a, h0, reverse=reverse)
        check_close(got, oracle(x, a, h0, lens, reverse), x, a, h0, lens, reverse, 'cfg3')
    # bitwise: forward and all three gradients
    x, a, h0, ls = _inputs(lens, (64,), torch.float32, seed=13, initial=True)
    g = torch.randn_like(x)
    outs = []
    for _ in range(2):
        y, grads = _grads(lambda u, v, w: rua.segment_linear_recurrence(u, ls, v, w), (x, a, h0), g)
        outs.append((y,) + tuple(grads))
    for u, v in zip(*outs):
        assert torch.equal(u, v)
