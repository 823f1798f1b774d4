"""Per-sequence prefix scans (segment_cumsum / logcumsumexp / cummax / cummin and the layout methods) against torch's own
scans applied to every sequence on the same GPU: floats through fp64 upcasts, max / min in the storage dtype."""
import numpy as np
import pytest
import torch

import torchrua_b200 as rua

pytestmark = pytest.mark.gpu

DEV = torch.device('cuda')
DTYPES = [torch.float32, torch.float64, torch.float16, torch.bfloat16]
OPS = ['sum', 'logsumexp', 'max', 'min']
LAYOUTS = ['C', 'L', 'P', 'R']
TORCH = {'sum': torch.cumsum, 'logsumexp': torch.logcumsumexp, 'max': torch.cummax, 'min': torch.cummin}
FREE = {'sum': rua.segment_cumsum, 'logsumexp': rua.segment_logcumsumexp, 'max': rua.segment_cummax,
        'min': rua.segment_cummin}
METHOD = {'sum': 'cumsum', 'logsumexp': 'logcumsumexp', 'max': 'cummax', 'min': 'cummin'}


def _data(lens, feat, dtype, seed=0, ties=False):
    g = torch.Generator().manual_seed(seed)
    n = int(sum(lens))
    x = torch.randn((n,) + tuple(feat), generator=g, dtype=torch.float64)
    if ties:
        x = torch.randint(-3, 4, x.shape, generator=g).double()
    return x.to(dtype).to(DEV), torch.tensor(lens, dtype=torch.long, device=DEV)


def _rev_rows(lens):
    """C row of token (i, len-1-t) for every C row (i, t)"""
    lens = torch.as_tensor(lens, dtype=torch.long)
    off = torch.cumsum(lens, 0) - lens
    seg = torch.repeat_interleave(torch.arange(lens.numel()), lens)
    t = torch.arange(int(lens.sum())) - off[seg]
    return (off[seg] + lens[seg] - 1 - t).to(DEV), t.to(DEV), lens[seg].to(DEV)


def oracle(op, x, lens, reverse):
    """torch scan per sequence in C order: (values, indices or None).  Padding after the tokens never influences a prefix,
    so one padded call along dim 1 gives every sequence's scan."""
    rrows, t, seg_len = _rev_rows(lens)
    if reverse:
        x = x[rrows]
    w = x.double() if op in ('sum', 'logsumexp') else x
    B, T = len(lens), max(list(lens) + [1])
    pad = torch.zeros((B, T) + tuple(x.shape[1:]), dtype=w.dtype, device=DEV)
    seg = torch.repeat_interleave(torch.arange(B, device=DEV), torch.as_tensor(lens, device=DEV))
    pad[seg, t] = w
    res = TORCH[op](pad, dim=1)
    if op in ('max', 'min'):
        v, i = res.values[seg, t], res.indices[seg, t]
        if reverse:
            v, i = v[rrows], i[rrows]
            i = seg_len.view((-1,) + (1,) * (i.dim() - 1)) - 1 - i
        return v, i
    y = res[seg, t]
    return (y[rrows] if reverse else y), None


def global_prefix(x, lens, reverse):
    """per-sequence running sum in fp64 as a global prefix minus its value before each sequence (no padding)"""
    rrows, _, _ = _rev_rows(lens)
    xr = x.double()[rrows] if reverse else x.double()
    glob = torch.cumsum(xr, 0)
    ls = torch.as_tensor(lens, device=DEV)
    seg = torch.repeat_interleave(torch.arange(len(lens), device=DEV), ls)
    base = torch.cat([torch.zeros_like(glob[:1]), glob])[(torch.cumsum(ls, 0) - ls)[seg]]
    out = glob - base
    return out[rrows] if reverse else out


def prefix_abs(x, lens, reverse):
    return global_prefix(x.abs(), lens, reverse)


def check_close(op, got, ref, x, lens, reverse):
    scale = prefix_abs(x, lens, reverse)
    if op == 'logsumexp':
        scale = scale + 1
    if x.dtype == torch.float64:
        tol = 1e-12
    elif x.dtype == torch.float32:
        tol = 1e-5
    else:
        tol = 1e-2
        ref = ref.to(x.dtype).double()   # the fp32 computation rounded once
    err = (got.double() - ref).abs()
    bound = tol * ref.abs() + tol * scale
    bad = ~(err <= bound) & ~(torch.isinf(ref) & (got.double() == ref))
    assert not bad.any(), f'{op} {x.dtype}: max err {err[bad].max().item()} at {bad.nonzero()[:4].tolist()}'


def check_exact(got_v, got_i, ref_v, ref_i):
    assert torch.equal(torch.isnan(got_v), torch.isnan(ref_v))
    assert torch.equal(got_v.nan_to_num(0.0), ref_v.nan_to_num(0.0))
    assert torch.equal(got_i, ref_i)


def make_layout(kind, x, lens, extra_width=0, fill=0.0):
    c = rua.C(data=x, token_sizes=lens)
    if kind == 'C':
        return c
    if kind == 'P':
        return c.pack()
    z = c.left(fill) if kind == 'L' else c.right(fill)
    if extra_width:
        b = z.data.shape[0]
        pad = torch.full((b, extra_width) + tuple(x.shape[1:]), 7.0, dtype=x.dtype, device=DEV)
        data = torch.cat([z.data, pad], 1) if kind == 'L' else torch.cat([pad, z.data], 1)
        z = z._replace(data=data)
    return z


def run_layout(kind, op, x, lens, reverse, extra_width=0):
    z = make_layout(kind, x, lens, extra_width)
    res = getattr(z, METHOD[op])(reverse=reverse)
    if op in ('max', 'min'):
        v, i = res
        return z, v, i, v.cat().data, i.cat().data
    return z, res, None, res.cat().data, None


SHAPES = [([3, 0, 5, 1, 7, 2, 0], (8,)), ([1], (3,)), ([4, 9, 0, 6], (1,)), ([40, 3, 17, 0, 2], (1024,)),
          ([5, 0, 3, 8], (4, 5)), ([0, 0], (8,))]


@pytest.mark.parametrize('reverse', [False, True])
@pytest.mark.parametrize('kind', LAYOUTS)
@pytest.mark.parametrize('dtype', DTYPES)
@pytest.mark.parametrize('op', OPS)
def test_forward_parity(op, dtype, kind, reverse):
    for k, (lens, feat) in enumerate(SHAPES):
        x, ls = _data(lens, feat, dtype, seed=k, ties=op in ('max', 'min') and k % 2 == 0)
        _, _, _, got, got_i = run_layout(kind, op, x, ls, reverse)
        ref, ref_i = oracle(op, x, lens, reverse)
        if op in ('max', 'min'):
            check_exact(got, got_i, ref, ref_i)
        else:
            check_close(op, got, ref, x, lens, reverse)
        free = FREE[op](x, ls, reverse=reverse)
        if op in ('max', 'min'):
            check_exact(free.values, free.indices, ref, ref_i)
        else:
            check_close(op, free, ref, x, lens, reverse)


def test_ties_and_nan_follow_torch():
    x = torch.tensor([1, 3, 3, 2, float('nan'), 5, float('nan')], device=DEV)
    lens = torch.tensor([7], device=DEV)
    for op in ('max', 'min'):
        for reverse in (False, True):
            got = FREE[op](x, lens, reverse=reverse)
            ref_v, ref_i = oracle(op, x, [7], reverse)
            check_exact(got.values, got.indices, ref_v, ref_i)
    assert rua.segment_cummax(x, lens).indices.tolist() == [0, 1, 2, 2, 4, 4, 6]


@pytest.mark.parametrize('dtype', [torch.float32, torch.float64])
def test_long_sequences_across_many_chunks(dtype):
    lens = [1, 4096, 0, 70000, 3]
    for op in OPS:
        if op in ('sum', 'logsumexp') and dtype == torch.float32:
            continue   # a 70000-term fp32 running sum drifts past 1e-5 of sum |x| by itself; fp64 checks the carries
        x, ls = _data(lens, (4,), dtype, seed=3, ties=op in ('max', 'min'))
        for reverse in (False, True):
            for kind in LAYOUTS:
                _, _, _, got, got_i = run_layout(kind, op, x, ls, reverse)
                ref, ref_i = oracle(op, x, lens, reverse)
                if op in ('max', 'min'):
                    check_exact(got, got_i, ref, ref_i)
                else:
                    check_close(op, got, ref, x, lens, reverse)


def cfg3_lengths(B=16384, seed=0):
    rng = np.random.default_rng(seed)
    return np.minimum(rng.zipf(1.5, B), 4096).tolist()


def test_cfg3_lengths_cumsum_and_determinism():
    lens = cfg3_lengths()
    x, ls = _data(lens, (64,), torch.float32, seed=5)
    for reverse in (False, True):
        got = rua.segment_cumsum(x, ls, reverse=reverse)
        check_close('sum', got, global_prefix(x, lens, reverse), x, lens, reverse)
    # determinism: forward and backward of every op, bitwise
    for op in OPS:
        outs = []
        for _ in range(2):
            xx = x.clone().requires_grad_(True)
            res = FREE[op](xx, ls)
            y = res.values if op in ('max', 'min') else res
            (g,) = torch.autograd.grad(y, xx, torch.ones_like(y) * 0.5)
            outs.append((y.detach(), g))
        assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1]), op


@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16])
@pytest.mark.parametrize('H', [1, 2, 4])
def test_narrow_rows(dtype, H):
    rng = np.random.default_rng(H)
    lens = rng.integers(1, 64, 32768)
    lens[::97] = 0
    lens[5000] = 1500
    lens[20000] = 4000
    lens = lens.tolist() + [0, 0, 0]
    for op in OPS:
        x, ls = _data(lens, (H,), dtype, seed=H, ties=op in ('max', 'min'))
        got = FREE[op](x, ls)
        ref, ref_i = oracle(op, x, lens, False)
        if op in ('max', 'min'):
            check_exact(got.values, got.indices, ref, ref_i)
        else:
            check_close(op, got, ref, x, lens, False)


@pytest.mark.parametrize('kind', ['L', 'R'])
@pytest.mark.parametrize('op', OPS)
def test_padding_rows_copied_through(kind, op):
    lens = [3, 0, 5, 2]
    x, ls = _data(lens, (8,), torch.float32, seed=1)
    z, out, idx, got, _ = run_layout(kind, op, x, ls, False, extra_width=3)
    mask = rua.C(data=torch.ones(len(x), 1, device=DEV), token_sizes=ls)
    tok = (mask.left(0) if kind == 'L' else mask.right(0)).data[..., 0] > 0
    tok = torch.cat([tok, torch.zeros(len(lens), 3, dtype=torch.bool, device=DEV)], 1) if kind == 'L' else \
        torch.cat([torch.zeros(len(lens), 3, dtype=torch.bool, device=DEV), tok], 1)
    assert torch.equal(out.data[~tok], z.data[~tok])
    if idx is not None:
        assert (idx.data[~tok] == 0).all()
    data = z.data.clone().requires_grad_(True)
    res = getattr(z._replace(data=data), METHOD[op])()
    y = (res[0] if op in ('max', 'min') else res).data
    g = torch.randn_like(y)
    (gx,) = torch.autograd.grad(y, data, g)
    assert torch.equal(gx[~tok], g[~tok])


def test_cat_rows_past_the_tokens():
    lens = [3, 4]
    x, _ = _data([3, 4, 5], (8,), torch.float32, seed=2)   # 12 rows, the segments cover 7
    ls = torch.tensor(lens, device=DEV)
    for op in OPS:
        xx = x.clone().requires_grad_(True)
        res = FREE[op](xx, ls)
        y = res.values if op in ('max', 'min') else res
        assert torch.equal(y[7:].detach(), x[7:])
        if op in ('max', 'min'):
            assert (res.indices[7:] == 0).all()
        g = torch.randn_like(y)
        (gx,) = torch.autograd.grad(y, xx, g)
        assert torch.equal(gx[7:], g[7:])
        ref, ref_i = oracle(op, x[:7], lens, False)
        if op in ('max', 'min'):
            check_exact(y[:7].detach(), res.indices[:7], ref, ref_i)
        else:
            check_close(op, y[:7].detach(), ref, x[:7], lens, False)


@pytest.mark.parametrize('kind', LAYOUTS)
@pytest.mark.parametrize('op', OPS)
def test_reverse_equals_rev_scan_rev(kind, op):
    lens = [5, 0, 9, 1, 4]
    x, ls = _data(lens, (16,), torch.float32, seed=4, ties=op in ('max', 'min'))
    z = make_layout(kind, x, ls)
    a = getattr(z, METHOD[op])(reverse=True)
    b = getattr(z.rev(), METHOD[op])()
    if op in ('max', 'min'):
        assert torch.equal(a[0].cat().data, b[0].rev().cat().data)
        lenrow = _rev_rows(lens)[2].view(-1, 1)
        assert torch.equal(a[1].cat().data, lenrow - 1 - b[1].rev().cat().data)
    else:
        torch.testing.assert_close(a.cat().data, b.rev().cat().data, rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize('kind', LAYOUTS)
@pytest.mark.parametrize('op', OPS)
def test_gradcheck_fp64(kind, op):
    lens = [3, 0, 4, 1]
    x, ls = _data(lens, (3,), torch.float64, seed=6)
    z = make_layout(kind, x, ls)
    for reverse in (False, True):
        def f(d):
            res = getattr(z._replace(data=d), METHOD[op])(reverse=reverse)
            return (res[0] if op in ('max', 'min') else res).data
        assert torch.autograd.gradcheck(f, (z.data.clone().requires_grad_(True),))


@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16])
@pytest.mark.parametrize('op', OPS)
def test_gradients_against_torch(op, dtype):
    lens = [6, 0, 11, 1, 300]
    x, ls = _data(lens, (32,), dtype, seed=7)
    for reverse in (False, True):
        xx = x.clone().requires_grad_(True)
        res = FREE[op](xx, ls, reverse=reverse)
        y = res.values if op in ('max', 'min') else res
        g = torch.randn_like(y)
        (got,) = torch.autograd.grad(y, xx, g)
        # torch autograd of the per-sequence op (fp64 for the smooth ops)
        xr = x.double() if op in ('sum', 'logsumexp') else x
        xr = xr.clone().requires_grad_(True)
        off = [0] + np.cumsum(lens).tolist()
        outs = []
        for i, n in enumerate(lens):
            seq = xr[off[i]:off[i + 1]]
            seq = seq.flip(0) if reverse else seq
            r = TORCH[op](seq, 0)
            r = r.values if op in ('max', 'min') else r
            outs.append(r.flip(0) if reverse else r)
        (ref,) = torch.autograd.grad(torch.cat(outs), xr, g.to(xr.dtype))
        tol = 1e-4 if dtype == torch.float32 else 3e-2
        torch.testing.assert_close(got.double(), ref.double(), rtol=tol, atol=tol * (1 + ref.abs().max().item()))


def test_cummax_gradient_lands_on_returned_index():
    x = torch.tensor([[1.], [3.], [3.], [2.], [3.], [0.]], device=DEV, requires_grad=True)
    lens = torch.tensor([6], device=DEV)
    for op, fn in (('max', rua.segment_cummax), ('min', rua.segment_cummin)):
        res = fn(x, lens)
        (g,) = torch.autograd.grad(res.values, x, torch.ones_like(res.values))
        want = torch.zeros(6, device=DEV)
        want.index_add_(0, res.indices[:, 0], torch.ones(6, device=DEV))
        assert torch.equal(g[:, 0], want)


def test_cumsum_double_backward_and_others_raise():
    lens = [4, 0, 7]
    x, ls = _data(lens, (5,), torch.float64, seed=8)
    xx = x.clone().requires_grad_(True)
    y = rua.segment_cumsum(xx, ls)
    (g,) = torch.autograd.grad((y ** 2).sum(), xx, create_graph=True)
    (gg,) = torch.autograd.grad((g ** 2).sum(), xx)
    xr = x.clone().requires_grad_(True)
    yr = torch.cat([torch.cumsum(s, 0) for s in torch.split(xr, lens)])
    (gr,) = torch.autograd.grad((yr ** 2).sum(), xr, create_graph=True)
    (ggr,) = torch.autograd.grad((gr ** 2).sum(), xr)
    torch.testing.assert_close(gg, ggr)
    for op in ('logsumexp', 'max', 'min'):
        xx = x.clone().requires_grad_(True)
        res = FREE[op](xx, ls)
        y = res.values if op in ('max', 'min') else res
        (g,) = torch.autograd.grad(y.sum(), xx, create_graph=True)
        with pytest.raises(RuntimeError):
            torch.autograd.grad(g.sum(), xx)


def test_logcumsumexp_minus_inf_gradient():
    x = torch.tensor([[-float('inf')], [0.], [1.], [-float('inf')], [2.]], device=DEV, dtype=torch.float64,
                     requires_grad=True)
    lens = torch.tensor([3, 2], device=DEV)
    y = rua.segment_logcumsumexp(x, lens)
    (g,) = torch.autograd.grad(y.sum(), x)
    assert g[0, 0] == 0 and g[3, 0] == 0
    # the finite positions get torch's gradient of the finite part
    xr = torch.tensor([0., 1.], dtype=torch.float64, requires_grad=True)
    (gr,) = torch.autograd.grad(torch.logcumsumexp(xr, 0).sum(), xr)
    torch.testing.assert_close(g[1:3, 0], gr.to(DEV))
    assert torch.allclose(g[4, 0], torch.tensor(1.0, dtype=torch.float64, device=DEV))


def test_layout_results_keep_metadata():
    lens = [3, 0, 5]
    x, ls = _data(lens, (4,), torch.float32, seed=9)
    for kind in LAYOUTS:
        z = make_layout(kind, x, ls)
        for m in METHOD.values():
            res = getattr(z, m)()
            for r in (res if isinstance(res, tuple) and not hasattr(res, 'data') else (res,)):
                assert type(r) is type(z)
                if kind == 'P':
                    assert r.batch_sizes is z.batch_sizes and r.sorted_indices is z.sorted_indices
                    assert r.unsorted_indices is z.unsorted_indices
                else:
                    assert r.token_sizes is z.token_sizes
