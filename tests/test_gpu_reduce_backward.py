"""Gradients of the six segment reductions on every backward kernel path (csrc/reduce_bwd.cu, csrc/reduce_warpseg_bwd.cu)
against fp64 references computed on the same GPU with plain torch ops, vectorised over segment ids.

Each case is checked two ways:
- formula on the stored output: the documented gradient (include/rua_b200.h) evaluated in fp64 on the inputs x, the
  cotangent g and the kernel's own forward output.  fp64 within 1e-12, fp32 within 1e-5 (+ 1e-6 |g|), fp16 / bf16
  faithfully rounded (the fp64 value rounded either way: one ulp); sum bit-equal to g; max / min put a non-zero gradient
  on exactly the rows equal to the output.
- true gradient: the fp64 gradient of the fp64 reduction (softmax for logsumexp, the exact product of the other rows for
  prod), allowing for the rounding of the stored output and the forward's accumulation.

Every case names the path its shape selects; test_every_case_runs_the_kernel_it_names confirms it from the profiler.
Rows that no segment owns (sum of sizes < N) and a batch of zero segments get a zero gradient."""
import re

import numpy as np
import pytest
import torch

import torchrua_b200 as rua
from torchrua_b200 import _native
from tests.test_gpu_warpseg import S_MIN, SIZES as WARPSEG_SIZES

pytestmark = pytest.mark.gpu

DEV = torch.device('cuda')
F64, F32, F16, BF16 = torch.float64, torch.float32, torch.float16, torch.bfloat16
DTYPES = [F64, F32, F16, BF16]
OPS = ['sum', 'mean', 'prod', 'max', 'min', 'logsumexp']
OP_CODE = {op: i for i, op in enumerate(OPS)}                  # enum rua_reduce_op
VEC = {F64: 2, F32: 4, F16: 8, BF16: 8}                        # elements per 16-byte vector
CTYPE = {F64: 'double', F32: 'float', F16: '__half', BF16: '__nv_bfloat16'}
MANT = {F16: 10, BF16: 7}                                      # explicit mantissa bits
U_ACC = {F64: 2.0 ** -53, F32: 2.0 ** -24, F16: 2.0 ** -24, BF16: 2.0 ** -24}   # unit roundoff of the accumulator
RTOL = {F64: 1e-12, F32: 1e-5, F16: 1e-2, BF16: 1e-2}


def _dn(dtype):
    return {F64: 'f64', F32: 'f32', F16: 'f16', BF16: 'bf16'}[dtype]


def _long(r):        # long segments (N > 8 S) with an empty, a one-row and a 1500-row segment
    return np.concatenate([r.integers(100, 700, 24), [0, 1, 1500, 0, 2]])


def _tiles(r):
    return np.concatenate([r.integers(0, 150, 20), [1, 400, 0]])


def _pieces(r):      # sub-word pieces (N <= 8 S) with giants that cross many chunks
    return np.concatenate([r.integers(1, 5, 1500), [3000], r.integers(1, 5, 1500), [4500, 0, 1], r.integers(1, 5, 1000),
                           [5000]])


def _case(path, dtype, H, sizes, tail=0, shift=0, inline=False, wide=False, sum_loss=False):
    return dict(path=path, dtype=dtype, H=H, sizes=sizes, tail=tail, shift=shift, inline=inline, wide=wide,
                sum_loss=sum_loss)


# id -> case.  path: 'warpseg' (segreduce_bwd_warpseg_kernel) or the V of segreduce_bwd_kernel; inline: max / min take
# the INLINE instance with tie_count_crossing_kernel.  fp64 / fp16 cases carry rows past the last segment.
CASES = {}
for _dt in DTYPES:
    _t = 5 if _dt in (F64, F16) else 0
    for _name in sorted(WARPSEG_SIZES):                      # H = 1, >= 32768 segments, aligned
        CASES[f'warpseg-{_name}-{_dn(_dt)}'] = _case('warpseg', _dt, 1, WARPSEG_SIZES[_name], tail=_t,
                                                     wide=_name == 'long_among_short', sum_loss=_name == 'all_ones')
    CASES[f'vec-{_dn(_dt)}'] = _case(VEC[_dt], _dt, 64 * VEC[_dt], _long, tail=_t, wide=True)   # 32 <= H/V <= 256
    CASES[f'tiles257-{_dn(_dt)}'] = _case(VEC[_dt], _dt, 257 * VEC[_dt], _tiles, tail=_t)     # partial last tile
    CASES[f'shortrow-{_dn(_dt)}'] = _case(VEC[_dt], _dt, {F64: 6, F32: 24, F16: 16, BF16: 8}[_dt], _long, tail=_t,
                                          sum_loss=True)                                     # H/V < 32
    CASES[f'odd7-{_dn(_dt)}'] = _case(1, _dt, 7, _long, tail=_t)
    CASES[f'misaligned-{_dn(_dt)}'] = _case(1, _dt, 64, _long, tail=_t, shift=1)            # H % V == 0, base off by 1
    CASES[f'pieces-{_dn(_dt)}'] = _case(VEC[_dt], _dt, {F64: 64, F32: 128, F16: 8, BF16: 256}[_dt], _pieces, tail=_t,
                                        inline=True)
CASES['tiles512-bf16'] = _case(8, BF16, 4096, _tiles)
CASES['odd301-bf16'] = _case(1, BF16, 301, _long)
CASES['odd301-f32'] = _case(1, F32, 301, _long, tail=3)
CASES['misaligned-scalars-f32'] = _case(1, F32, 1, WARPSEG_SIZES['cfg5_like'], shift=1)   # warpseg shape, unaligned


# ---------------------------------------------------------------------------------------------------------------------
# inputs
# ---------------------------------------------------------------------------------------------------------------------
def draw(op, dtype, shape, seg_first, lens_rows, seed, wide=False, order=None):
    """payload for `op` (float64 before the cast): ties for max / min, values near 1 with zeros for prod, a wide range and
    -inf entries for logsumexp.  Row order[k] (k when order is None) is the k-th row in segment order, where every
    segment's rows are contiguous; seg_first[k]: it is the first row of its segment, lens_rows[k]: its segment's length
    (0 for rows no segment owns)."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    n = shape[0]
    pos = torch.arange(n, device=DEV)
    first = pos[seg_first]
    ln = lens_rows[first]
    row = (lambda k: k) if order is None else (lambda k: order[k])   # noqa: E731
    if op in ('max', 'min'):
        return torch.randint(-3, 4, shape, generator=g, device=DEV).to(F64).to(dtype)
    if op == 'logsumexp':
        if wide and dtype in (F64, F32):
            x = torch.rand(shape, generator=g, device=DEV, dtype=F64) * 2000 - 1000
        else:
            x = torch.randn(shape, generator=g, device=DEV, dtype=F64) * 3
        # -inf on 3 % of the rows, also leading a segment; the last row of every segment stays finite.  The longest
        # segment starts with 40 of them: whole batches of rows before the first finite value.
        minf = torch.rand(n, generator=g, device=DEV) < 0.03
        lead = first[ln.argmax()]
        minf[row(pos[lead:lead + min(40, int(ln.max()) - 1)])] = True
        minf[row(first + ln - 1)] = False
        x[minf] = float('-inf')
        return x.to(dtype)
    if op == 'prod':
        x = torch.exp(torch.randn(shape, generator=g, device=DEV, dtype=F64) * 0.02)
        x = torch.where(torch.rand(shape, generator=g, device=DEV) < 0.5, -x, x)
        x = x.to(dtype)
        # one zero in every 7th segment of >= 2 rows (at its middle), two zeros in every 11th of >= 3 (first and last),
        # every 13th one-row segment is a zero, and the longest segment has a zero in its middle
        mid = first + ln // 2
        pick = torch.cat([mid[ln >= 2][::7], first[ln >= 3][3::11], (first + ln - 1)[ln >= 3][3::11], first[ln == 1][::13],
                          mid[ln.argmax()].view(1)])
        x[row(pick)] = 0
        return x
    return torch.randn(shape, generator=g, device=DEV, dtype=F64).to(dtype)


def cotangent(S, feat, dtype, seed):
    """signed, |g| in [0.5, 2): a tie count never rounds g / n to zero"""
    g = torch.Generator(device=DEV).manual_seed(seed)
    mag = torch.rand((S,) + feat, generator=g, device=DEV, dtype=F64) * 1.5 + 0.5
    sign = torch.where(torch.rand((S,) + feat, generator=g, device=DEV) < 0.5, -1.0, 1.0)
    return (mag * sign.to(F64)).to(dtype)


def segment_ids(lens, n_rows):
    """segment of every row, -1 past the last segment"""
    S = lens.numel()
    seg = torch.repeat_interleave(torch.arange(S, device=DEV), lens)
    return torch.cat([seg, torch.full((n_rows - seg.numel(),), -1, dtype=torch.long, device=DEV)])


def inputs(cid, op, extra_tail=0):
    """(x, sizes, seg, g) for case `cid`; x is a contiguous view `shift` elements into its buffer"""
    c = CASES[cid]
    dtype, H = c['dtype'], c['H']
    sizes = np.asarray(c['sizes'](np.random.default_rng(11)), dtype=np.int64)
    lens = torch.from_numpy(sizes).to(DEV)
    n = int(sizes.sum())
    N = n + c['tail'] + extra_tail
    feat = () if H == 1 else (H,)
    seg = segment_ids(lens, N)
    first = torch.zeros(N, dtype=torch.bool, device=DEV)
    first[(torch.cumsum(lens, 0) - lens)[lens > 0]] = True
    lens_rows = torch.where(seg >= 0, lens[seg.clamp_min(0)], 0)
    body = draw(op, dtype, (N,) + feat, first, lens_rows, seed=OP_CODE[op] + 17, wide=c['wide'])
    if c['shift']:
        buf = torch.empty(N * H + c['shift'], dtype=dtype, device=DEV)
        x = buf[c['shift']:].view((N,) + feat)
        x.copy_(body)
    else:
        x = body
    g = cotangent(len(sizes), feat, dtype, seed=OP_CODE[op] + 101)
    return x, lens, seg, g


# ---------------------------------------------------------------------------------------------------------------------
# reference and checks
# ---------------------------------------------------------------------------------------------------------------------
def _per_seg(vals, seg, S):
    return torch.zeros((S,) + vals.shape[1:], dtype=vals.dtype, device=DEV).index_add_(0, seg, vals)


def lse64(xs, sg, S):
    m = torch.full((S, xs.shape[1]), float('-inf'), dtype=F64, device=DEV).index_reduce_(0, sg, xs, 'amax')
    return m + torch.log(_per_seg(torch.exp(xs - m[sg]), sg, S))


def reference(op, x, seg, S, g, out):
    """(formula on the stored output, true fp64 gradient) on the rows some segment owns; everything (rows, H) fp64"""
    own = seg >= 0
    xs, sg = x[own], seg[own]
    gs, os = g[sg], out[sg]
    lens = torch.bincount(sg, minlength=S).to(F64).view(-1, 1)
    if op == 'sum':
        return gs, gs
    if op == 'mean':
        f = gs / lens[sg]
        return f, f
    if op in ('max', 'min'):
        eq = xs == os
        n = _per_seg(eq.to(F64), sg, S)
        f = torch.where(eq, gs / n[sg].clamp_min(1), 0.0)
        return f, f
    if op == 'logsumexp':
        return gs * torch.exp(xs - os), gs * torch.exp(xs - lse64(xs, sg, S)[sg])
    # prod: the product of the other rows from per-segment zero counts, signs and sum of log |x|
    zero = xs == 0
    nz = _per_seg(zero.to(F64), sg, S)[sg]
    neg = _per_seg((xs < 0).to(F64), sg, S)[sg] - (xs < 0).to(F64)
    logs = _per_seg(torch.where(zero, 0.0, torch.log(xs.abs())), sg, S)[sg] - torch.where(zero, 0.0, torch.log(xs.abs()))
    others = torch.where(nz - zero.to(F64) > 0, 0.0, torch.exp(logs) * (1 - 2 * torch.remainder(neg, 2)))
    true = gs * others
    return torch.where(zero, true, gs * os / torch.where(zero, 1.0, xs)), true


def ulp(a, dtype):
    """spacing of `dtype` at |a| (fp64 tensor)"""
    p = MANT[dtype]
    u = torch.ldexp(torch.ones_like(a), torch.frexp(a).exponent - 1 - p)
    return u.clamp_min(torch.finfo(dtype).tiny * 2.0 ** -p)


def bits(t):
    return t.contiguous().view({8: torch.int64, 4: torch.int32, 2: torch.int16}[t.element_size()])


def check(op, dtype, x, seg, g, out, grad, what):
    """grad (N, ...) against the fp64 references; rows no segment owns must be exactly 0"""
    N, S = x.shape[0], g.shape[0]
    x64, g64, o64 = (t.reshape(t.shape[0], -1).to(F64) for t in (x, g, out))
    got_all = grad.reshape(N, -1)
    own = seg >= 0
    assert bool((got_all[~own] == 0).all()), f'{what}: rows past the last segment are not 0'
    got = got_all[own]
    gd = got.to(F64)
    sg = seg[own]
    if op == 'logsumexp':     # the forward output the gradient is built on (-inf entries, also leading a run, add 0)
        lse, has = lse64(x64[own], sg, S), torch.bincount(sg, minlength=S) > 0
        fbad = ~((o64 - lse).abs()[has] <= RTOL[dtype] * (lse.abs()[has] + 1))     # a NaN output fails too
        assert not bool(fbad.any()), f'{what}: forward logsumexp off the fp64 value in {int(fbad.sum())} elements'
    assert not bool(gd.isnan().any()), f'{what}: NaN in the gradient'
    f, true = reference(op, x64, seg, S, g64, o64)
    gs, os = g64[sg], o64[sg]
    xs = x64[own]
    lens = torch.bincount(sg, minlength=S).to(F64).view(-1, 1)[sg]
    err = (gd - f).abs()
    if op == 'sum':
        assert torch.equal(bits(got), bits(g.reshape(S, -1)[sg])), f'{what}: sum gradient is not g broadcast, bit for bit'
    if op in ('max', 'min'):
        hit = (got != 0) == (xs == os)
        assert bool(hit.all()), f'{what}: {int((~hit).sum())} rows with a non-zero gradient differ from the tie rows'
    slack = torch.where(xs == 0, lens * U_ACC[dtype], 0.0) if op == 'prod' else 0.0   # the product of the others: len roundings
    if dtype in (F16, BF16):
        bound = ulp(torch.maximum(f.abs(), gd.abs()), dtype) + slack * f.abs()
    else:
        bound = (RTOL[dtype] + slack) * f.abs() + (1e-6 * gs.abs() if dtype == F32 else 1e-300)
    bad = err > bound
    assert not bool(bad.any()), \
        f'{what}: formula on the stored output: {int(bad.sum())} elements off, worst excess {float((err - bound).max()):.3g}'
    if op == 'logsumexp':
        minf = xs == float('-inf')
        assert bool((got[minf] == 0).all()), f'{what}: -inf entries must get exactly 0'
    if op in ('logsumexp', 'prod'):
        eps = torch.finfo(dtype).eps
        rel = RTOL[dtype] + lens * U_ACC[dtype] + (os.abs() * eps if op == 'logsumexp' else eps)
        bound = rel * true.abs() + 1e-6 * gs.abs()
        terr = (gd - true).abs()
        bad = terr > bound
        assert not bool(bad.any()), \
            f'{what}: true gradient: {int(bad.sum())} elements off, worst excess {float((terr - bound).max()):.3g}'


# ---------------------------------------------------------------------------------------------------------------------
# the backward paths
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('op', OPS)
@pytest.mark.parametrize('cid', sorted(CASES))
def test_gradient(cid, op):
    c = CASES[cid]
    if c['inline'] and op not in ('max', 'min'):
        pytest.skip('the INLINE instances exist for max / min only; the other ops of this shape run in vec-*')
    x, lens, seg, g = inputs(cid, op)
    leaf = x.detach().requires_grad_(True)              # keeps the view's (possibly unaligned) storage offset
    out = getattr(rua, 'segment_' + op)(leaf, lens)
    if c['sum_loss']:                                   # grad_out is a stride-0 expansion of ones
        out.sum().backward()
        g = torch.ones_like(out)
    else:
        out.backward(g)
    grad = leaf.grad
    check(op, c['dtype'], x, seg, g, out.detach(), grad, f'{cid} {op}')
    # deterministic: the C entry point again, on a buffer full of NaN, gives the same bits on every row
    again = torch.full_like(x, float('nan'))
    off = torch.cat([torch.zeros(1, dtype=torch.long, device=DEV), torch.cumsum(lens, 0)])
    _native._reduce_backward_raw(g.contiguous(), out.detach(), x, off, lens.numel(), OP_CODE[op], again)
    assert torch.equal(bits(again), bits(grad)), f'{cid} {op}: two backward runs differ'


@pytest.mark.parametrize('cid', sorted(CASES))
def test_rows_no_segment_owns_get_zero(cid):
    """rua_segment_reduce_backward writes all N rows: those at or past sum(sizes) come back 0 in a NaN-filled buffer"""
    for op in OPS:
        x, lens, seg, g = inputs(cid, op, extra_tail=7)
        off = torch.cat([torch.zeros(1, dtype=torch.long, device=DEV), torch.cumsum(lens, 0)])
        out = _native._reduce_raw(x.contiguous(), off, lens.numel(), OP_CODE[op])
        grad = torch.full_like(x, float('nan'))
        _native._reduce_backward_raw(g, out, x, off, lens.numel(), OP_CODE[op], grad)
        n = int(lens.sum())
        assert bool((grad[n:] == 0).all()), f'{cid} {op}: rows past the last segment are not 0'
        assert not bool(grad[:n].isnan().any()), f'{cid} {op}: a row of a segment was not written'


_KERNEL = re.compile(r'(segreduce_bwd_warpseg_kernel|segreduce_bwd_kernel|tie_count_crossing_kernel|tie_count_kernel)'
                     r'<([^<>]*)>')


def expected_kernels(cid, op):
    c = CASES[cid]
    t, k = CTYPE[c['dtype']], OP_CODE[op]
    if c['path'] == 'warpseg':
        return {f'segreduce_bwd_warpseg_kernel<{t},1,{k}>'}
    v, inline = c['path'], c['inline'] and op in ('max', 'min')
    want = {f'segreduce_bwd_kernel<{t},{v},{k},{str(inline).lower()}>'}
    if op in ('max', 'min'):
        want.add(f"{'tie_count_crossing_kernel' if inline else 'tie_count_kernel'}<{t},{v},{k}>")
    return want


def test_every_case_runs_the_kernel_it_names():
    """each case's backward, under the profiler, launches exactly the instances its path names"""
    from torch.profiler import ProfilerActivity, profile
    seen_any = False
    for cid in sorted(CASES):
        ops = ['max', 'min'] if CASES[cid]['inline'] else OPS
        runs = []
        for op in ops:
            x, lens, seg, g = inputs(cid, op)
            off = torch.cat([torch.zeros(1, dtype=torch.long, device=DEV), torch.cumsum(lens, 0)])
            out = _native._reduce_raw(x.contiguous(), off, lens.numel(), OP_CODE[op])
            runs.append((op, x, off, lens.numel(), g, out, torch.empty_like(x)))
        torch.cuda.synchronize()
        want = set()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for op, x, off, S, g, out, grad in runs:
                _native._reduce_backward_raw(g, out, x, off, S, OP_CODE[op], grad)
                want |= expected_kernels(cid, op)
            torch.cuda.synchronize()
        got = set()
        for e in prof.events():
            m = _KERNEL.search(e.name)
            if m:
                got.add(f'{m.group(1)}<{m.group(2).replace(" ", "")}>')
        seen_any = seen_any or bool(got)
        assert got, f'{cid}: the profiler captured no backward kernel'
        assert got == want, f'{cid}: launched {sorted(got)}, expected {sorted(want)}'
    assert seen_any


# ---------------------------------------------------------------------------------------------------------------------
# gathered rows: scatter_*, P.seg, L.seg
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('op', OPS)
@pytest.mark.parametrize('dtype,H,M', [(F32, 1, S_MIN + 7000), (BF16, 1, S_MIN + 7000), (BF16, 64, 3000)])
def test_scatter_gradient(op, dtype, H, M):
    """scatter_*(zeros, index, source): the backward runs on the source rows gathered in bucket order (the warp-per-32-
    segments kernel at H = 1); the reference applies per row with its bucket as the segment"""
    K = 6 * M
    index = torch.randint(0, M, (K,), generator=torch.Generator(device=DEV).manual_seed(3), device=DEV)
    lens = torch.bincount(index, minlength=M)
    feat = () if H == 1 else (H,)
    srt = torch.sort(index, stable=True).indices          # the source rows bucket by bucket
    first = torch.zeros(K, dtype=torch.bool, device=DEV)
    first[(torch.cumsum(lens, 0) - lens)[lens > 0]] = True
    src = draw(op, dtype, (K,) + feat, first, lens[index[srt]], seed=OP_CODE[op] + 29, order=srt)
    leaf = src.clone().requires_grad_(True)
    out = getattr(rua, 'scatter_' + op)(torch.zeros((M,) + feat, dtype=dtype, device=DEV), index, leaf)
    g = cotangent(M, feat, dtype, seed=OP_CODE[op] + 31)
    out.backward(g)
    check(op, dtype, src, index, g, out.detach(), leaf.grad, f'scatter_{op} {dtype} H={H}')


def _nested(dtype, H, op, seed):
    """a C of B sequences and a C of sub-segment sizes splitting every sequence (some sizes 0)"""
    r = np.random.default_rng(seed)
    lens = r.integers(1, 200, 64)
    dur, counts = [], []
    for ln in lens:
        cuts = np.sort(r.integers(0, ln + 1, r.integers(0, 12)))
        parts = np.diff(np.concatenate([[0], cuts, [ln]]))
        dur.append(parts)
        counts.append(len(parts))
    dur = torch.from_numpy(np.concatenate(dur)).to(DEV)
    lens_t, counts_t = torch.from_numpy(lens).to(DEV), torch.tensor(counts, device=DEV)
    n = int(lens.sum())
    seg = segment_ids(dur, n)
    first = torch.zeros(n, dtype=torch.bool, device=DEV)
    first[(torch.cumsum(dur, 0) - dur)[dur > 0]] = True
    x = draw(op, dtype, (n, H), first, dur[seg], seed=OP_CODE[op] + 43)
    return rua.C(data=x, token_sizes=lens_t), rua.C(data=dur, token_sizes=counts_t), seg


@pytest.mark.parametrize('op', OPS)
@pytest.mark.parametrize('dtype,H', [(F32, 24), (BF16, 64)])
def test_pack_seg_gradient(op, dtype, H):
    c, duration, seg = _nested(dtype, H, op, seed=5)
    code = rua.C(data=torch.arange(c.data.shape[0], device=DEV), token_sizes=c.token_sizes).pack().data   # P row -> C row
    leaf = c.data[code].clone().requires_grad_(True)
    p = c.pack()._replace(data=leaf)
    res = p.seg(duration, getattr(rua, 'segment_' + op))
    g = cotangent(duration.data.numel(), (H,), dtype, seed=OP_CODE[op] + 47)
    res.data.backward(duration._replace(data=g).pack().data)
    grad_c = torch.empty_like(leaf.grad)
    grad_c[code] = leaf.grad
    check(op, dtype, c.data, seg, g, res.cat().data.detach(), grad_c, f'P.seg {op} {dtype}')


@pytest.mark.parametrize('op', OPS)
@pytest.mark.parametrize('dtype,H', [(F32, 24), (BF16, 64)])
def test_left_seg_gradient(op, dtype, H):
    c, duration, seg = _nested(dtype, H, op, seed=6)
    left = c.left(0)
    leaf = left.data.clone().requires_grad_(True)
    res = left._replace(data=leaf).seg(duration, getattr(rua, 'segment_' + op))
    g = cotangent(duration.data.numel(), (H,), dtype, seed=OP_CODE[op] + 53)
    res.data.backward(duration._replace(data=g).left(0).data)
    B, T = leaf.shape[:2]
    lens = c.token_sizes
    b = torch.repeat_interleave(torch.arange(B, device=DEV), lens)
    t = torch.arange(c.data.shape[0], device=DEV) - (torch.cumsum(lens, 0) - lens)[b]
    flat = leaf.grad.reshape(B * T, H)
    tok = b * T + t
    pad = torch.ones(B * T, dtype=torch.bool, device=DEV)
    pad[tok] = False
    assert bool((flat[pad] == 0).all()), f'L.seg {op}: padding rows get a gradient'
    check(op, dtype, c.data, seg, g, res.cat().data.detach(), flat[tok], f'L.seg {op} {dtype}')


# ---------------------------------------------------------------------------------------------------------------------
# rows no segment owns, through the public API; zero segments
# ---------------------------------------------------------------------------------------------------------------------
def _dirty(like):
    """hand the allocator a NaN-filled block of this size: the next allocation of that size reuses it"""
    junk = torch.full_like(like, float('nan'))
    del junk


@pytest.mark.parametrize('op', OPS)
@pytest.mark.parametrize('shape', ['warpseg', 'chunk'])
def test_public_rows_past_the_segments(op, shape):
    """segment_* with sizes that cover only part of the rows, and C.seg on a C whose storage has rows past its tokens"""
    r = np.random.default_rng(9)
    if shape == 'warpseg':
        sizes, feat = r.integers(1, 5, S_MIN + 100), ()
    else:
        sizes, feat = r.integers(0, 40, 300), (32,)
    n = int(sizes.sum())
    N = n + 50
    lens = torch.from_numpy(sizes).to(DEV)
    seg = segment_ids(lens, N)
    first = torch.zeros(N, dtype=torch.bool, device=DEV)
    first[(torch.cumsum(lens, 0) - lens)[lens > 0]] = True
    x = draw(op, F32, (N,) + feat, first, torch.where(seg >= 0, lens[seg.clamp_min(0)], 0), seed=OP_CODE[op] + 61)
    g = cotangent(len(sizes), feat, F32, seed=OP_CODE[op] + 67)
    fn = getattr(rua, 'segment_' + op)
    leaf = x.clone().requires_grad_(True)
    out = fn(leaf, lens)
    _dirty(x)
    out.backward(g)
    check(op, F32, x, seg, g, out.detach(), leaf.grad, f'segment_{op} {shape}, short sizes')
    # C.seg: 7 sequences, each split into a run of the sub-segments `sizes`; the C holds n tokens in N rows
    owner = torch.arange(len(sizes), device=DEV) // ((len(sizes) + 6) // 7)
    per_seq = torch.zeros(7, dtype=torch.long, device=DEV).index_add_(0, owner, lens)
    counts = torch.bincount(owner, minlength=7)
    c = rua.C(data=x.clone().requires_grad_(True), token_sizes=per_seq)
    res = c.seg(rua.C(data=lens, token_sizes=counts), fn)
    _dirty(x)
    res.data.backward(g)
    check(op, F32, x, seg, g, res.data.detach(), c.data.grad, f'C.seg {op} {shape}, rows past the tokens')


@pytest.mark.parametrize('op', OPS)
@pytest.mark.parametrize('dtype', [F32, BF16])
def test_zero_segments(op, dtype):
    """no segment at all: the forward gives (0, *feat) and every row's gradient is 0, through the API and the C entry"""
    x = torch.randn(40, 3, device=DEV).to(dtype)
    leaf = x.clone().requires_grad_(True)
    out = getattr(rua, 'segment_' + op)(leaf, torch.zeros(0, dtype=torch.long, device=DEV))
    assert out.shape == (0, 3)
    _dirty(x)
    out.sum().backward()
    assert bool((leaf.grad == 0).all())
    grad = torch.full_like(x, float('nan'))
    off = torch.zeros(1, dtype=torch.long, device=DEV)
    empty = torch.empty(0, 3, dtype=dtype, device=DEV)
    _native._reduce_backward_raw(empty, empty, x, off, 0, OP_CODE[op], grad)
    assert bool((grad == 0).all())
