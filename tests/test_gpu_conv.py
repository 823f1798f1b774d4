"""Per-sequence depthwise 1-D convolution (segment_depthwise_conv1d and the layout methods) against F.conv1d(groups=H) in
fp64 on the same GPU, applied to every sequence zero-padded with p rows before and K - 1 - p after."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import torchrua_b200 as rua

pytestmark = pytest.mark.gpu

DEV = torch.device('cuda')
DTYPES = [torch.float32, torch.float64, torch.float16, torch.bfloat16]
LAYOUTS = ['C', 'L', 'P', 'R']
PADDINGS = ['causal', 'same', 0]
KS = [1, 2, 4, 31, 32]
SHAPES = [([3, 0, 5, 1, 7, 2, 0, 40], (1,)), ([1, 4, 9, 33], (3,)), ([6, 0, 35, 2], (1024,)), ([5, 0, 3, 8], (4, 5))]


def pad_of(padding, K):
    return K - 1 if padding == 'causal' else ((K - 1) // 2 if padding == 'same' else padding)


def _data(lens, feat, K, dtype, seed=0, bias=True):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn((int(sum(lens)),) + tuple(feat), generator=g, dtype=torch.float64)
    w = torch.randn(tuple(feat) + (K,), generator=g, dtype=torch.float64)
    b = torch.randn(tuple(feat), generator=g, dtype=torch.float64) if bias else None
    to = lambda t: None if t is None else t.to(dtype).to(DEV)   # noqa: E731
    return to(x), torch.tensor(lens, dtype=torch.long, device=DEV), to(w), to(b)


def oracle(x, lens, w, b, pad):
    """fp64 F.conv1d(groups=H) per sequence on the zero-padded (B, H, T) form with explicit F.pad(p, K - 1 - p)"""
    lens = [int(n) for n in lens]
    feat = tuple(x.shape[1:])
    H, K = int(np.prod(feat)), w.shape[-1]
    B, T = len(lens), max(lens + [1])
    ls = torch.tensor(lens, device=DEV)
    seg = torch.repeat_interleave(torch.arange(B, device=DEV), ls)
    t = torch.arange(x.shape[0], device=DEV) - (torch.cumsum(ls, 0) - ls)[seg]
    dense = torch.zeros(B, T, H, dtype=torch.float64, device=DEV)
    dense[seg, t] = x.double().reshape(-1, H)
    inp = F.pad(dense.transpose(1, 2), (pad, K - 1 - pad))
    y = F.conv1d(inp, w.double().reshape(H, 1, K), None if b is None else b.double().reshape(H), groups=H)
    return y.transpose(1, 2)[seg, t].reshape((-1,) + feat)


def check_close(got, x, lens, w, b, pad):
    ref = oracle(x, lens, w, b, pad)
    scale = oracle(x.abs(), lens, w.abs(), None if b is None else b.abs(), pad)
    if x.dtype == torch.float64:
        tol = 1e-12
    elif x.dtype == torch.float32:
        tol = 1e-5
    else:
        tol = 1e-2
        ref = ref.to(x.dtype).double()   # the fp64 result rounded once
    err = (got.double() - ref).abs()
    bad = ~(err <= tol * ref.abs() + tol * scale)
    assert not bad.any(), f'{x.dtype}: max err {err[bad].max().item()} at {bad.nonzero()[:4].tolist()}'


def make_layout(kind, x, lens, extra_width=0):
    c = rua.C(data=x, token_sizes=lens)
    if kind == 'C':
        return c
    if kind == 'P':
        return c.pack()
    z = c.left(0) if kind == 'L' else c.right(0)
    if extra_width:
        b = z.data.shape[0]
        pad = torch.full((b, extra_width) + tuple(x.shape[1:]), 7.0, dtype=x.dtype, device=DEV)
        z = z._replace(data=torch.cat([z.data, pad], 1) if kind == 'L' else torch.cat([pad, z.data], 1))
    return z


@pytest.mark.parametrize('kind', LAYOUTS)
@pytest.mark.parametrize('dtype', DTYPES)
def test_forward_parity(dtype, kind):
    for s, (lens, feat) in enumerate(SHAPES):
        for K in KS:
            for padding in PADDINGS:
                for bias in (True, False):
                    x, ls, w, b = _data(lens, feat, K, dtype, seed=s * 100 + K, bias=bias)
                    z = make_layout(kind, x, ls)
                    got = z.depthwise_conv1d(w, b, padding=padding)
                    assert type(got) is type(z)
                    check_close(got.cat().data, x, lens, w, b, pad_of(padding, K))
                    if kind == 'C':
                        free = rua.segment_depthwise_conv1d(x, ls, w, b, padding=padding)
                        assert torch.equal(free, got.data)


@pytest.mark.parametrize('kind', LAYOUTS)
@pytest.mark.parametrize('dtype', [torch.float64, torch.float32])
def test_gradients_against_oracle(dtype, kind):
    lens, feat = [6, 0, 11, 1, 70, 3], (24,)
    for K, padding in ((4, 'causal'), (31, 'same'), (5, 1), (8, 0)):
        x, ls, w, b = _data(lens, feat, K, dtype, seed=K)
        z = make_layout(kind, x, ls)
        data, ww, bb = z.data.clone().requires_grad_(True), w.clone().requires_grad_(True), b.clone().requires_grad_(True)
        y = z._replace(data=data).depthwise_conv1d(ww, bb, padding=padding)
        g = torch.randn_like(y.data)
        gd, gw, gb = torch.autograd.grad(y.data, (data, ww, bb), g)
        # the oracle in fp64 on the C rows, gradient of the same loss
        gc = y._replace(data=g).cat().data
        xr, wr, br = (t.double().clone().requires_grad_(True) for t in (x, w, b))
        yr = oracle(xr, lens, wr, br, pad_of(padding, K))
        rx, rw, rb = torch.autograd.grad(yr, (xr, wr, br), gc.double())
        got_x = z._replace(data=gd).cat().data
        tol = 1e-10 if dtype == torch.float64 else 1e-4
        for got, ref in ((got_x, rx), (gw, rw), (gb, rb)):
            torch.testing.assert_close(got.double(), ref, rtol=tol, atol=tol * (1 + ref.abs().max().item()))


@pytest.mark.parametrize('kind', LAYOUTS)
def test_gradcheck_fp64(kind):
    lens = [3, 0, 4, 1]
    for K, padding in ((3, 'causal'), (4, 'same'), (2, 0)):
        x, ls, w, b = _data(lens, (3,), K, torch.float64, seed=6)
        z = make_layout(kind, x, ls)

        def f(d, ww, bb):
            return z._replace(data=d).depthwise_conv1d(ww, bb, padding=padding).data
        assert torch.autograd.gradcheck(f, (z.data.clone().requires_grad_(True), w.clone().requires_grad_(True),
                                            b.clone().requires_grad_(True)))


def test_frozen_weight_and_input_without_grad():
    lens = [5, 0, 9, 2]
    x, ls, w, b = _data(lens, (16,), 4, torch.float32, seed=3)
    xx = x.clone().requires_grad_(True)
    y = rua.segment_depthwise_conv1d(xx, ls, w, b, padding='causal')   # frozen weight and bias
    (gx,) = torch.autograd.grad(y, xx, torch.ones_like(y))
    ww = w.clone().requires_grad_(True)
    y2 = rua.segment_depthwise_conv1d(x, ls, ww, None, padding='causal')   # input without grad
    (gw,) = torch.autograd.grad(y2, ww, torch.ones_like(y2))
    xr, wr = x.double().requires_grad_(True), w.double().requires_grad_(True)
    yr = oracle(xr, lens, wr, None, 3)
    rx, rw = torch.autograd.grad(yr, (xr, wr), torch.ones_like(yr))
    torch.testing.assert_close(gx.double(), rx, rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(gw.double(), rw, rtol=1e-5, atol=1e-4)


def test_double_backward_raises():
    x, ls, w, b = _data([4, 7], (5,), 3, torch.float64, seed=8)
    xx = x.clone().requires_grad_(True)
    y = rua.segment_depthwise_conv1d(xx, ls, w, b, padding='same')
    (g,) = torch.autograd.grad((y ** 2).sum(), xx, create_graph=True)
    with pytest.raises(RuntimeError):
        torch.autograd.grad(g.sum(), xx)


@pytest.mark.parametrize('dtype', [torch.float32, torch.float64])
def test_long_sequence_across_many_chunks(dtype):
    lens = [1, 70000, 0, 3, 5000]
    for K, padding in ((4, 'causal'), (31, 'same'), (32, 0)):
        x, ls, w, b = _data(lens, (4,), K, dtype, seed=K)
        for kind in LAYOUTS:
            got = make_layout(kind, x, ls).depthwise_conv1d(w, b, padding=padding).cat().data
            check_close(got, x, lens, w, b, pad_of(padding, K))


@pytest.mark.parametrize('H', [1, 2])
@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16])
def test_many_short_sequences_narrow_rows(dtype, H):
    rng = np.random.default_rng(H)
    lens = rng.integers(1, 64, 32768)
    lens[::97] = 0
    lens[5000] = 1500
    lens = lens.tolist() + [0, 0, 0]
    for K, padding in ((4, 'causal'), (31, 'same')):
        x, ls, w, b = _data(lens, (H,), K, dtype, seed=H)
        check_close(rua.segment_depthwise_conv1d(x, ls, w, b, padding=padding), x, lens, w, b, pad_of(padding, K))
        xx = x.clone().requires_grad_(True)
        y = rua.segment_depthwise_conv1d(xx, ls, w, b, padding=padding)
        (gx,) = torch.autograd.grad(y, xx, torch.ones_like(y))
        xr = x.double().requires_grad_(True)
        yr = oracle(xr, lens, w, b, pad_of(padding, K))
        (rx,) = torch.autograd.grad(yr, xr, torch.ones_like(yr))
        tol = 1e-4 if dtype == torch.float32 else 3e-2
        torch.testing.assert_close(gx.double(), rx, rtol=tol, atol=tol * (1 + rx.abs().max().item()))


@pytest.mark.parametrize('kind', ['L', 'R'])
def test_padding_rows_copied_through(kind):
    lens = [3, 0, 5, 2]
    x, ls, w, b = _data(lens, (8,), 4, torch.float32, seed=1)
    z = make_layout(kind, x, ls, extra_width=3)
    mask = rua.C(data=torch.ones(len(x), 1, device=DEV), token_sizes=ls)
    tok = (mask.left(0) if kind == 'L' else mask.right(0)).data[..., 0] > 0
    extra = torch.zeros(len(lens), 3, dtype=torch.bool, device=DEV)
    tok = torch.cat([tok, extra], 1) if kind == 'L' else torch.cat([extra, tok], 1)
    data, ww, bb = z.data.clone().requires_grad_(True), w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    out = z._replace(data=data).depthwise_conv1d(ww, bb, padding='same')
    assert torch.equal(out.data[~tok].detach(), z.data[~tok])
    check_close(out.cat().data.detach(), x, lens, w, b, 1)
    g = torch.randn_like(out.data)
    gx, gw, gb = torch.autograd.grad(out.data, (data, ww, bb), g)
    assert torch.equal(gx[~tok], g[~tok])
    gc = (rua.L if kind == 'L' else rua.R)(data=g[:, :-3] if kind == 'L' else g[:, 3:], token_sizes=ls).cat().data
    wr, br = w.double().requires_grad_(True), b.double().requires_grad_(True)
    yr = oracle(x, lens, wr, br, 1)
    rw, rb = torch.autograd.grad(yr, (wr, br), gc.double())
    torch.testing.assert_close(gw.double(), rw, rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(gb.double(), rb, rtol=1e-4, atol=1e-4)


def test_cat_rows_past_the_tokens():
    lens = [3, 4]
    x, _, w, b = _data([3, 4, 5], (8,), 4, torch.float32, seed=2)   # 12 rows, the segments cover 7
    ls = torch.tensor(lens, device=DEV)
    xx = x.clone().requires_grad_(True)
    y = rua.segment_depthwise_conv1d(xx, ls, w, b, padding='causal')
    assert torch.equal(y[7:].detach(), x[7:])
    check_close(y[:7].detach(), x[:7], lens, w, b, 3)
    g = torch.randn_like(y)
    (gx,) = torch.autograd.grad(y, xx, g)
    assert torch.equal(gx[7:], g[7:])


def test_cfg3_lengths():
    lens = np.minimum(np.random.default_rng(0).zipf(1.5, 16384), 4096).tolist()
    for K, padding in ((4, 'causal'), (31, 'same')):
        x, ls, w, b = _data(lens, (4,), K, torch.float32, seed=5)   # the dense fp64 oracle is B x 4096 x H
        check_close(rua.segment_depthwise_conv1d(x, ls, w, b, padding=padding), x, lens, w, b, pad_of(padding, K))


def test_determinism_with_thousands_of_chunks():
    lens = np.random.default_rng(1).integers(1, 300, 2000).tolist()
    for dtype in (torch.float32, torch.bfloat16):
        for K, padding in ((4, 'causal'), (31, 'same')):
            x, ls, w, b = _data(lens, (256,), K, dtype, seed=9)
            outs = []
            for _ in range(2):
                xx, ww, bb = (t.clone().requires_grad_(True) for t in (x, w, b))
                y = rua.segment_depthwise_conv1d(xx, ls, ww, bb, padding=padding)
                grads = torch.autograd.grad(y, (xx, ww, bb), torch.ones_like(y) * 0.5)
                outs.append((y.detach(),) + grads)
            for a, c in zip(*outs):
                assert torch.equal(a, c)


@pytest.mark.parametrize('kind', ['C', 'P', 'L'])
@pytest.mark.parametrize('dtype,feat', [(torch.float32, (256,)), (torch.float32, (67,)), (torch.bfloat16, (512,))])
def test_merged_gradients_many_chunks(dtype, feat, kind):
    """forward, grad_in, grad_weight and grad_bias against the fp64 oracle where every CTA walks many chunks and the
    weight / bias partials of hundreds of slots and several column blocks are merged (16-byte and one-element rows)"""
    lens = np.random.default_rng(2).integers(1, 300, 2000).tolist()
    tol = 1e-4 if dtype == torch.float32 else 1e-2
    for K, padding in ((4, 'causal'), (31, 'same')):
        x, ls, w, b = _data(lens, feat, K, dtype, seed=K)
        z = make_layout(kind, x, ls)
        data, ww, bb = z.data.clone().requires_grad_(True), w.clone().requires_grad_(True), b.clone().requires_grad_(True)
        y = z._replace(data=data).depthwise_conv1d(ww, bb, padding=padding)
        check_close(y.cat().data.detach(), x, lens, w, b, pad_of(padding, K))
        g = torch.randn(y.data.shape, generator=torch.Generator(device=DEV).manual_seed(K), device=DEV).to(dtype)
        got = torch.autograd.grad(y.data, (data, ww, bb), g)
        got = (z._replace(data=got[0]).cat().data,) + got[1:]
        gc = y._replace(data=g).cat().data.double()
        p = pad_of(padding, K)
        xr, wr, br = (t.double().requires_grad_(True) for t in (x, w, b))
        ref = torch.autograd.grad(oracle(xr, lens, wr, br, p), (xr, wr, br), gc)
        # sum |g| |x| (weight), sum |w| |g| (input), sum |g| (bias): the scale of each accumulated entry
        xa, wa, ba = (t.double().abs().requires_grad_(True) for t in (x, w, b))
        scale = torch.autograd.grad(oracle(xa, lens, wa, ba, p), (xa, wa, ba), gc.abs())
        for name, gv, rv, sv in zip(('grad_in', 'grad_weight', 'grad_bias'), got, ref, scale):
            if dtype != torch.float32:
                rv = rv.to(dtype).double()   # the fp64 result rounded once
            err = (gv.double() - rv).abs()
            bad = ~(err <= tol * rv.abs() + tol * sv)
            assert not bad.any(), f'{name} K={K}: max err {err[bad].max().item()} at {bad.nonzero()[:4].tolist()}'


def test_constant_lengths_equal_dense_conv1d():
    B, T, H = 6, 50, 40
    for K, padding in ((4, 'causal'), (7, 'same'), (5, 0)):
        x, ls, w, b = _data([T] * B, (H,), K, torch.float32, seed=K)
        z = rua.C(data=x, token_sizes=ls).left(0)
        got = z.depthwise_conv1d(w, b, padding=padding).data
        p = pad_of(padding, K)
        want = F.conv1d(F.pad(z.data.transpose(1, 2), (p, K - 1 - p)), w.view(H, 1, K), b, groups=H).transpose(1, 2)
        torch.testing.assert_close(got, want, rtol=1e-5, atol=1e-5)


def test_results_keep_metadata():
    x, ls, w, b = _data([3, 0, 5], (4,), 3, torch.float32, seed=9)
    for kind in LAYOUTS:
        z = make_layout(kind, x, ls)
        r = z.depthwise_conv1d(w, b, padding='causal')
        assert type(r) is type(z)
        if kind == 'P':
            assert r.batch_sizes is z.batch_sizes and r.sorted_indices is z.sorted_indices
            assert r.unsorted_indices is z.unsorted_indices
        else:
            assert r.token_sizes is z.token_sizes
