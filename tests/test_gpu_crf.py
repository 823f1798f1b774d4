"""Linear-chain CRF (torchrua_b200.crf) against an fp64 oracle on the same GPU.

The oracle is the forward algorithm on the zero-padded (B, T, K) batch, a loop over T vectorised over B and masked by
length; its gradients come from autograd.  Viterbi is the same loop in max-plus with smallest-index ties, plus a
backtrack.  The oracle itself is checked against brute-force enumeration of every path.

Tolerances (u = unit roundoff of the accumulator: fp32 for fp32 / fp16 / bf16, fp64 for fp64; m = max|x| + max|W| +
max|start| + max|end|): log Z, the best score and the log-likelihood within 16 u (|ref| + len (1 + m)), where |ref| is
|log Z| + |score| for the log-likelihood; grad_x within |g| (1e-5 + 16 u len (1 + m)), plus one ulp of the storage dtype
for 16-bit inputs; grad_W / grad_start / grad_end within the same per-term bound times sum_i |g_i| len_i.  The bound is
tight enough to catch one missing or doubled step at T = 4096 (a step moves log Z by about log K + m).
"""
import itertools
import math

import numpy as np
import pytest
import torch

import torchrua_b200 as rua

pytestmark = pytest.mark.gpu

DEV = 'cuda'
DTYPES = [torch.float32, torch.float64, torch.float16, torch.bfloat16]
ULP = {torch.float16: 2.0 ** -10, torch.bfloat16: 2.0 ** -7}


def _u(dtype):
    return 2.0 ** -53 if dtype == torch.float64 else 2.0 ** -24


# ---------------------------------------------------------------------------------------------------------------------
# fp64 oracle
# ---------------------------------------------------------------------------------------------------------------------
def pad(x, lens):
    """(N, K) C rows -> zero-padded (B, T, K) through plain torch indexing (differentiable)."""
    B = lens.numel()
    T = int(lens.max()) if B else 0
    off = torch.cumsum(lens, 0) - lens
    t = torch.arange(T, device=x.device)
    valid = t[None, :] < lens[:, None]
    idx = (off[:, None] + t[None, :]).clamp(max=max(x.shape[0] - 1, 0))
    return torch.where(valid[..., None], x[idx], torch.zeros((), dtype=x.dtype, device=x.device)), valid


def _zero(K, ref):
    return torch.zeros(K, dtype=ref.dtype, device=ref.device)


def oracle_log_z(x, lens, W, start=None, end=None):
    xp, valid = pad(x, lens)
    K = x.shape[-1]
    start = _zero(K, x) if start is None else start
    end = _zero(K, x) if end is None else end
    B, T = valid.shape
    if T == 0:
        return torch.zeros(B, dtype=x.dtype, device=x.device)
    alpha = start + xp[:, 0]
    for t in range(1, T):
        nxt = torch.logsumexp(alpha[:, :, None] + W[None], dim=1) + xp[:, t]
        alpha = torch.where(valid[:, t, None], nxt, alpha)
    lz = torch.logsumexp(alpha + end, dim=1)
    return torch.where(lens > 0, lz, torch.zeros_like(lz))


def oracle_score(x, lens, tags, W, start=None, end=None):
    xp, valid = pad(x, lens)
    yp, _ = pad(tags[:, None], lens)
    y = yp[..., 0].clamp(0, x.shape[-1] - 1)
    K = x.shape[-1]
    start = _zero(K, x) if start is None else start
    end = _zero(K, x) if end is None else end
    B, T = valid.shape
    if T == 0:
        return torch.zeros(B, dtype=x.dtype, device=x.device)
    s = torch.where(valid, xp.gather(2, y[..., None])[..., 0], torch.zeros((), dtype=x.dtype, device=x.device)).sum(1)
    tr = W[y[:, :-1], y[:, 1:]]
    s = s + torch.where(valid[:, 1:], tr, torch.zeros((), dtype=x.dtype, device=x.device)).sum(1)
    last = y.gather(1, (lens - 1).clamp(min=0)[:, None])[:, 0]
    s = s + start[y[:, 0]] + end[last]
    return torch.where(lens > 0, s, torch.zeros_like(s))


def oracle_viterbi(x, lens, W, start=None, end=None):
    """(tags in C rows, best score); max-plus with the smallest index winning every tie."""
    xp, valid = pad(x, lens)
    K = x.shape[-1]
    start = _zero(K, x) if start is None else start
    end = _zero(K, x) if end is None else end
    B, T = valid.shape
    if T == 0:
        return torch.empty(0, dtype=torch.long, device=x.device), torch.zeros(B, dtype=x.dtype, device=x.device)
    idx = torch.arange(K, device=x.device)
    alpha = start + xp[:, 0]
    bps = [None]
    for t in range(1, T):
        v = alpha[:, :, None] + W[None]
        best = v.max(dim=1).values
        arg = torch.where(v == best[:, None, :], idx[None, :, None], K).min(dim=1).values
        bps.append(arg)
        alpha = torch.where(valid[:, t, None], best + xp[:, t], alpha)
    fin = alpha + end
    top = fin.max(dim=1).values
    last = torch.where(fin == top[:, None], idx[None], K).min(dim=1).values
    ys = torch.full((B, T), -1, dtype=torch.long, device=x.device)
    y = last.clone()
    for t in range(T - 1, -1, -1):
        act = t < lens
        y = torch.where(t == lens - 1, last, y)
        ys[:, t] = torch.where(act, y, -1)
        if t > 0:
            y = torch.where(act, bps[t].gather(1, y[:, None])[:, 0], y)
    return ys[valid], torch.where(lens > 0, top, torch.zeros_like(top))


def scale_m(x, W, start, end):
    def mx(t):
        if t is None:
            return 0.0
        f = t.double()[torch.isfinite(t.double())]
        return float(f.abs().max()) if f.numel() else 0.0
    return mx(x) + mx(W) + mx(start) + mx(end)


def bound(ref, lens, m, dtype):
    return 16 * _u(dtype) * (ref.abs() + lens.double() * (1 + m))


def make(lens_list, K, dtype, ends=True, seed=0, scale=1.0, extra_rows=0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    lens = torch.tensor(lens_list, dtype=torch.long, device=DEV)
    N = int(lens.sum())
    x = (scale * torch.randn((N + extra_rows, K), generator=g, device=DEV, dtype=torch.float64)).to(dtype)
    W = torch.randn((K, K), generator=g, device=DEV, dtype=torch.float64).to(dtype)
    st = torch.randn(K, generator=g, device=DEV, dtype=torch.float64).to(dtype) if ends else None
    en = torch.randn(K, generator=g, device=DEV, dtype=torch.float64).to(dtype) if ends else None
    tags = torch.randint(0, K, (N + extra_rows,), generator=g, device=DEV)
    return lens, x, W, st, en, tags


def d64(t):
    return None if t is None else t.double()


def as_layout(kind, lens, x, fill=0):
    """(object of layout kind over the C rows x, function mapping that layout's (rows, ...) data back to C rows)"""
    c = rua.C(data=x, token_sizes=lens)
    if kind == 'C':
        return c, lambda d: d
    if kind == 'P':
        z = c.pack()
        return z, lambda d: z._replace(data=d).cat().data
    z = c.left(fill) if kind == 'L' else c.right(fill)
    return z, lambda d: type(z)(data=d, token_sizes=z.token_sizes).cat().data


# ---------------------------------------------------------------------------------------------------------------------
# the oracle itself
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('K,ends', [(1, True), (2, False), (2, True), (3, True)])
def test_oracle_matches_enumeration(K, ends):
    lens_list = [1, 2, 3, 4, 5, 0]
    lens, x, W, st, en, _ = make(lens_list, K, torch.float64, ends)
    lz = oracle_log_z(x, lens, W, st, en)
    vt, vbest = oracle_viterbi(x, lens, W, st, en)
    off = 0
    for i, n in enumerate(lens_list):
        if n == 0:
            assert lz[i] == 0 and vbest[i] == 0
            continue
        scores = []
        for path in itertools.product(range(K), repeat=n):
            p = torch.tensor(path, device=DEV)
            tags = torch.zeros(int(lens.sum()), dtype=torch.long, device=DEV)
            tags[off:off + n] = p
            scores.append(float(oracle_score(x, lens, tags, W, st, en)[i]))
        scores = np.array(scores)
        ref = np.logaddexp.reduce(scores)
        assert abs(float(lz[i]) - ref) <= 1e-12 * (1 + abs(ref))
        assert abs(np.exp(scores - float(lz[i])).sum() - 1) <= 1e-12        # sum_y exp(LL(y)) = 1
        assert abs(float(vbest[i]) - scores.max()) <= 1e-12 * (1 + abs(scores.max()))
        best_path = tuple(vt[off:off + n].tolist())
        assert abs(scores[list(itertools.product(range(K), repeat=n)).index(best_path)] - scores.max()) <= 1e-12
        off += n


# ---------------------------------------------------------------------------------------------------------------------
# the grid: dtype x layout x K x start / end, with empty and one-token sequences
# ---------------------------------------------------------------------------------------------------------------------
GRID_LENS = [0, 1, 3, 7, 2, 0, 13, 5, 1, 9, 33]


def check_forward(lz, ll, lens, x, W, st, en, tags, dtype):
    x64, W64, s64, e64 = d64(x), d64(W), d64(st), d64(en)
    m = scale_m(x, W, st, en)
    ref_lz = oracle_log_z(x64, lens, W64, s64, e64)
    assert lz.dtype == (torch.float64 if dtype == torch.float64 else torch.float32)
    err = (lz.double() - ref_lz).abs()
    assert bool((err <= bound(ref_lz, lens, m, dtype)).all()), (err.max(), ref_lz)
    if ll is not None:
        ref_sc = oracle_score(x64, lens, tags, W64, s64, e64)
        err = (ll.double() - (ref_sc - ref_lz)).abs()
        assert bool((err <= 16 * _u(dtype) * (ref_lz.abs() + ref_sc.abs() + lens.double() * (1 + m))).all())
    return ref_lz, m


@pytest.mark.parametrize('ends', [False, True])
@pytest.mark.parametrize('K', [1, 2, 5, 32, 33, 64])
@pytest.mark.parametrize('kind', ['C', 'L', 'P', 'R'])
@pytest.mark.parametrize('dtype', DTYPES, ids=str)
def test_grid(dtype, kind, K, ends):
    lens, x, W, st, en, tags = make(GRID_LENS, K, dtype, ends, seed=K)
    z, back = as_layout(kind, lens, x)
    zt, _ = as_layout(kind, lens, tags, fill=-100)
    # forward: log Z and the log-likelihood
    lz = z.crf_log_partition(W, st, en)
    ll = z.crf_log_likelihood(zt.data, W, st, en)
    ref_lz, m = check_forward(lz, ll, lens, x, W, st, en, tags, dtype)
    # decode: rescored path ~ oracle best, -1 on padding rows
    dec, best = z.crf_decode(W, st, en)
    assert type(dec) is type(z) and dec.data.dtype == torch.long and dec.data.shape == z.data.shape[:-1]
    path = back(dec.data)
    assert bool(((path >= 0) & (path < K)).all())
    if kind in ('L', 'R'):
        assert int((dec.data == -1).sum()) == dec.data.numel() - int(lens.sum())
    vt, vbest = oracle_viterbi(d64(x), lens, d64(W), d64(st), d64(en))
    tol = bound(vbest, lens, m, dtype)
    assert bool(((best.double() - vbest).abs() <= tol).all())
    rescored = oracle_score(d64(x), lens, path, d64(W), d64(st), d64(en))
    assert bool(((rescored - vbest).abs() <= tol).all())
    if dtype == torch.float64:
        assert torch.equal(path, vt)
    # gradients of sum_i g_i LL_i, all four inputs, through the layout's own storage
    g = torch.randn(lens.numel(), device=DEV, dtype=torch.float64)
    data = z.data.detach().requires_grad_(True)
    Wg = W.detach().requires_grad_(True)
    sg = None if st is None else st.detach().requires_grad_(True)
    eg = None if en is None else en.detach().requires_grad_(True)
    zz = z._replace(data=data)
    out = zz.crf_log_likelihood(zt.data, Wg, sg, eg)
    out.backward(g.to(out.dtype))
    xr = x.double().detach().requires_grad_(True)
    Wr = W.double().detach().requires_grad_(True)
    sr = None if st is None else st.double().detach().requires_grad_(True)
    er = None if en is None else en.double().detach().requires_grad_(True)
    ref = oracle_score(xr, lens, tags, Wr, sr, er) - oracle_log_z(xr, lens, Wr, sr, er)
    ref.backward(g)
    per_row = torch.repeat_interleave(g.abs() * (1e-5 + 16 * _u(dtype) * lens.double() * (1 + m)), lens)
    gx = back(data.grad).double()
    tol = per_row[:, None] + (ULP[dtype] * xr.grad.abs() + 2.0 ** -24 if dtype in ULP else 0)
    assert bool(((gx - xr.grad).abs() <= tol).all()), float((gx - xr.grad).abs().max())
    if kind in ('L', 'R'):
        pad_rows = data.grad.flatten(0, 1)[(dec.data == -1).flatten()]
        assert bool((pad_rows == 0).all())
    Lmax = int(lens.max())
    scale = (1e-5 + 16 * _u(dtype) * Lmax * (1 + m)) * float((g.abs() * lens.double()).sum())
    for got, want in ((Wg.grad, Wr.grad), (None if sg is None else sg.grad, None if sr is None else sr.grad),
                      (None if eg is None else eg.grad, None if er is None else er.grad)):
        if want is None:
            continue
        t = scale + (ULP[dtype] * want.abs() + 2.0 ** -24 if dtype in ULP else 0)
        assert bool(((got.double() - want).abs() <= t).all()), float((got.double() - want).abs().max())


def test_c_rows_past_the_tokens():
    """C storage with rows past sum(sizes): decode gives -1 there and grad_x gives 0."""
    lens, x, W, st, en, tags = make([3, 0, 4], 5, torch.float32, extra_rows=3)
    xs = x.detach().requires_grad_(True)
    rua.segment_crf_log_partition(xs, lens, W, st, en).sum().backward()
    assert bool((xs.grad[7:] == 0).all()) and bool((xs.grad[:7] != 0).any())
    out, best = rua.segment_crf_decode(x, lens, W, st, en)
    assert out[7:].tolist() == [-1, -1, -1] and bool((out[:7] >= 0).all())
    assert rua.C(data=x, token_sizes=lens).crf_decode(W)[0].data[7:].tolist() == [-1, -1, -1]


# ---------------------------------------------------------------------------------------------------------------------
# long sequences, many short ones, cfg3 lengths
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('kind', ['C', 'P'])
def test_long_sequences(kind):
    lens, x, W, st, en, tags = make([4100, 1, 0, 4096, 17, 4095], 5, torch.float32)
    z, back = as_layout(kind, lens, x)
    zt, _ = as_layout(kind, lens, tags)
    lz = z.crf_log_partition(W, st, en)
    ll = z.crf_log_likelihood(zt.data, W, st, en)
    ref_lz, m = check_forward(lz, ll, lens, x, W, st, en, tags, torch.float32)
    # one dropped or doubled step moves log Z by ~log K + x, far above the bound
    assert float(bound(ref_lz, lens, m, torch.float32).max()) < 0.5
    data = z.data.detach().requires_grad_(True)
    Wg = W.detach().requires_grad_(True)
    z._replace(data=data).crf_log_partition(Wg, st, en).sum().backward()
    xr, Wr = x.double().requires_grad_(True), W.double().requires_grad_(True)
    oracle_log_z(xr, lens, Wr, d64(st), d64(en)).sum().backward()
    per_row = torch.repeat_interleave(1e-5 + 16 * _u(torch.float32) * lens.double() * (1 + m), lens)
    assert bool(((back(data.grad).double() - xr.grad).abs() <= per_row[:, None]).all())
    scale = (1e-5 + 16 * _u(torch.float32) * 4100 * (1 + m)) * float(lens.sum())
    assert bool(((Wg.grad.double() - Wr.grad).abs() <= scale).all())
    _, best = z.crf_decode(W, st, en)
    _, vbest = oracle_viterbi(d64(x), lens, d64(W), d64(st), d64(en))
    assert bool(((best.double() - vbest).abs() <= bound(vbest, lens, m, torch.float32)).all())


def test_many_short_sequences():
    rng = np.random.default_rng(1)
    lens_list = rng.integers(0, 9, 40000).tolist()
    lens, x, W, st, en, tags = make(lens_list, 33, torch.float32, seed=3)
    xs, Wg = x.detach().requires_grad_(True), W.detach().requires_grad_(True)
    ll = rua.segment_crf_log_likelihood(xs, lens, tags, Wg, st, en)
    ref_lz, m = check_forward(rua.segment_crf_log_partition(x, lens, W, st, en), ll, lens, x, W, st, en, tags,
                              torch.float32)
    g = torch.randn(lens.numel(), device=DEV, dtype=torch.float64)
    ll.backward(g.float())
    xr, Wr = x.double().requires_grad_(True), W.double().requires_grad_(True)
    (oracle_score(xr, lens, tags, Wr, d64(st), d64(en)) - oracle_log_z(xr, lens, Wr, d64(st), d64(en))).backward(g)
    per_row = torch.repeat_interleave(g.abs() * (1e-5 + 16 * _u(torch.float32) * lens.double() * (1 + m)), lens)
    assert bool(((xs.grad.double() - xr.grad).abs() <= per_row[:, None]).all())
    scale = (1e-5 + 16 * _u(torch.float32) * 8 * (1 + m)) * float((g.abs() * lens.double()).sum())
    assert bool(((Wg.grad.double() - Wr.grad).abs() <= scale).all())


@pytest.mark.parametrize('kind', ['C', 'P'])
def test_cfg3_lengths(kind):
    lens_list = np.minimum(np.random.default_rng(0).zipf(1.5, 16384), 4096).tolist()
    lens, x, W, st, en, tags = make(lens_list, 5, torch.bfloat16, seed=4)
    z, _ = as_layout(kind, lens, x)
    zt, _ = as_layout(kind, lens, tags)
    check_forward(z.crf_log_partition(W, st, en), z.crf_log_likelihood(zt.data, W, st, en), lens, x, W, st, en, tags,
                  torch.bfloat16)
    m = scale_m(x, W, st, en)
    _, best = z.crf_decode(W, st, en)
    _, vbest = oracle_viterbi(d64(x), lens, d64(W), d64(st), d64(en))
    assert bool(((best.double() - vbest).abs() <= bound(vbest, lens, m, torch.bfloat16)).all())


# ---------------------------------------------------------------------------------------------------------------------
# robustness: -inf constraints, all paths forbidden, large emissions
# ---------------------------------------------------------------------------------------------------------------------
def bio(dtype):
    """tags O, B-X, I-X, B-Y, I-Y: I-X only after B-X / I-X, I-Y only after B-Y / I-Y, no I-* first"""
    K = 5
    W = torch.randn((K, K), generator=torch.Generator(device=DEV).manual_seed(7), device=DEV, dtype=torch.float64)
    for a in range(K):
        if a not in (1, 2):
            W[a, 2] = -math.inf
        if a not in (3, 4):
            W[a, 4] = -math.inf
    st = torch.zeros(K, device=DEV, dtype=torch.float64)
    st[2] = st[4] = -math.inf
    return W.to(dtype), st.to(dtype)


@pytest.mark.parametrize('dtype', DTYPES, ids=str)
def test_bio_constraints(dtype):
    W, st = bio(dtype)
    lens, x, _, _, en, tags = make([6, 1, 0, 40, 9], 5, dtype, seed=8)
    Wg, sg = W.detach().requires_grad_(True), st.detach().requires_grad_(True)
    xs = x.detach().requires_grad_(True)
    lz = rua.segment_crf_log_partition(xs, lens, Wg, sg, en)
    assert bool(torch.isfinite(lz).all())
    ref = oracle_log_z(d64(x), lens, d64(W), d64(st), d64(en))
    m = scale_m(x, W, st, en)
    assert bool(((lz.double() - ref).abs() <= bound(ref, lens, m, dtype)).all())
    lz.sum().backward()
    assert bool(torch.isfinite(xs.grad).all()) and bool(torch.isfinite(Wg.grad).all())
    assert bool((Wg.grad[torch.isinf(W)] == 0).all()) and bool((sg.grad[torch.isinf(st)] == 0).all())
    # marginals of forbidden first tags are exactly 0
    first = torch.cumsum(lens, 0) - lens
    rows = first[lens > 0]
    assert bool((xs.grad[rows][:, [2, 4]] == 0).all())
    out, best = rua.segment_crf_decode(x, lens, W, st, en)
    rescored = oracle_score(d64(x), lens, out, d64(W), d64(st), d64(en))
    assert bool(torch.isfinite(rescored).all())
    _, vbest = oracle_viterbi(d64(x), lens, d64(W), d64(st), d64(en))
    assert bool(((rescored - vbest).abs() <= bound(vbest, lens, m, dtype)).all())


@pytest.mark.parametrize('kind', ['C', 'L', 'P', 'R'])
def test_all_paths_forbidden(kind):
    lens, x, W, st, en, tags = make([4, 5, 3], 4, torch.float32, seed=9)
    x = x.clone()
    x[4 + 2] = -math.inf                  # every tag of the third token of sequence 1
    z, back = as_layout(kind, lens, x)
    data = z.data.detach().requires_grad_(True)
    Wg = W.detach().requires_grad_(True)
    lz = z._replace(data=data).crf_log_partition(Wg, st, en)
    assert lz[1].item() == -math.inf and bool(torch.isfinite(lz[[0, 2]]).all())
    lz[[0, 2]].sum().backward(retain_graph=True)
    g_ok = Wg.grad.clone()
    data.grad = None
    Wg.grad = None
    lz.backward(torch.ones(3, device=DEV))   # the -inf sequence contributes zero, not NaN
    gx = back(data.grad)
    assert bool((gx[4:9] == 0).all()) and bool(torch.isfinite(gx).all())
    assert torch.equal(Wg.grad, g_ok)


def test_large_emissions():
    """emissions x100: an exp-space recursion overflows or underflows here"""
    lens, x, W, st, en, tags = make([50, 7, 300, 1], 9, torch.float32, seed=10, scale=100.0)
    xs, Wg = x.detach().requires_grad_(True), W.detach().requires_grad_(True)
    lz = rua.segment_crf_log_partition(xs, lens, Wg, st, en)
    ref_lz, m = check_forward(lz, None, lens, x, W, st, en, tags, torch.float32)
    lz.sum().backward()
    xr, Wr = x.double().requires_grad_(True), W.double().requires_grad_(True)
    oracle_log_z(xr, lens, Wr, d64(st), d64(en)).sum().backward()
    per_row = torch.repeat_interleave(1e-5 + 16 * _u(torch.float32) * lens.double() * (1 + m), lens)
    assert bool(((xs.grad.double() - xr.grad).abs() <= per_row[:, None]).all())


# ---------------------------------------------------------------------------------------------------------------------
# decode ties, layouts, determinism, edge cases
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('dtype', DTYPES, ids=str)
@pytest.mark.parametrize('K', [2, 5, 33, 64])
def test_decode_ties_exact(dtype, K):
    g = torch.Generator(device=DEV).manual_seed(K)
    lens = torch.tensor([5, 0, 1, 12, 64, 3], device=DEV)
    N = int(lens.sum())
    x = torch.randint(-2, 3, (N, K), generator=g, device=DEV).to(dtype)
    W = torch.randint(-2, 3, (K, K), generator=g, device=DEV).to(dtype)
    st = torch.randint(-1, 2, (K,), generator=g, device=DEV).to(dtype)
    x[:3] = 0                                   # whole rows of ties
    vt, vbest = oracle_viterbi(d64(x), lens, d64(W), d64(st), None)
    for kind in ('C', 'L', 'P', 'R'):
        z, back = as_layout(kind, lens, x)
        dec, best = z.crf_decode(W, st)
        assert torch.equal(back(dec.data), vt), kind
        assert torch.equal(best.double(), vbest), kind


def test_layouts_bit_identical():
    lens, x, W, st, en, tags = make(GRID_LENS * 3, 33, torch.bfloat16, seed=11)
    g = torch.randn(lens.numel(), device=DEV)
    res = {}
    for kind in ('C', 'L', 'P', 'R'):
        z, back = as_layout(kind, lens, x)
        zt, _ = as_layout(kind, lens, tags, fill=-100)
        data = z.data.detach().requires_grad_(True)
        Wg, sg, eg = (t.detach().requires_grad_(True) for t in (W, st, en))
        ll = z._replace(data=data).crf_log_likelihood(zt.data, Wg, sg, eg)
        ll.backward(g)
        dec, best = z.crf_decode(W, st, en)
        res[kind] = (z.crf_log_partition(W, st, en), ll.detach(), back(dec.data), best, back(data.grad), Wg.grad,
                     sg.grad, eg.grad)
    for kind in ('L', 'P', 'R'):
        for a, b in zip(res['C'], res[kind]):
            assert torch.equal(a, b), kind


def test_repeated_runs_bit_identical():
    rng = np.random.default_rng(2)
    lens, x, W, st, en, tags = make(rng.integers(0, 300, 3000).tolist(), 64, torch.float32, seed=12)
    g = torch.randn(lens.numel(), device=DEV)

    def run():
        xs, Wg, sg, eg = (t.detach().requires_grad_(True) for t in (x, W, st, en))
        ll = rua.segment_crf_log_likelihood(xs, lens, tags, Wg, sg, eg)
        ll.backward(g)
        return (ll.detach(), *rua.segment_crf_decode(x, lens, W, st, en), xs.grad, Wg.grad, sg.grad, eg.grad)

    first = run()
    for _ in range(2):
        for a, b in zip(first, run()):
            assert torch.equal(a, b)


def test_out_of_range_tags_nan_for_that_sequence_only():
    lens, x, W, st, en, tags = make([3, 4, 2, 0], 6, torch.float32, seed=13)
    ok = rua.segment_crf_log_likelihood(x, lens, tags, W, st, en)
    for bad in (6, -1, 100):
        t = tags.clone()
        t[3 + 2] = bad                    # the third token of sequence 1
        ll = rua.segment_crf_log_likelihood(x, lens, t, W, st, en)
        assert math.isnan(ll[1].item())
        assert torch.equal(ll[[0, 2, 3]], ok[[0, 2, 3]])
    # tags at padding rows are ignored
    left = rua.C(data=x, token_sizes=lens).left(0)
    lt = rua.C(data=tags, token_sizes=lens).left(-100)
    assert torch.equal(left.crf_log_likelihood(lt.data, W, st, en), ok)


def test_empty_sequences_and_batches():
    lens, x, W, st, en, tags = make([0, 0, 2], 3, torch.float32, seed=14)
    xs, Wg = x.detach().requires_grad_(True), W.detach().requires_grad_(True)
    ll = rua.segment_crf_log_likelihood(xs, lens, tags, Wg, st, en)
    assert ll[:2].tolist() == [0.0, 0.0]
    assert rua.segment_crf_log_partition(x, lens, W, st, en)[:2].tolist() == [0.0, 0.0]
    assert rua.segment_crf_decode(x, lens, W, st, en)[1][:2].tolist() == [0.0, 0.0]
    # only empty sequences: zero gradients everywhere
    lens0 = torch.zeros(3, dtype=torch.long, device=DEV)
    x0 = torch.randn(0, 3, device=DEV, requires_grad=True)
    W0 = W.detach().requires_grad_(True)
    out = rua.segment_crf_log_partition(x0, lens0, W0, st, en)
    assert out.tolist() == [0.0, 0.0, 0.0]
    out.sum().backward()
    assert bool((W0.grad == 0).all())


def test_gradcheck_fp64():
    lens, x, W, st, en, tags = make([3, 0, 1, 4], 3, torch.float64, seed=15)
    args = tuple(t.detach().requires_grad_(True) for t in (x, W, st, en))
    assert torch.autograd.gradcheck(lambda a, b, c, d: rua.segment_crf_log_partition(a, lens, b, c, d), args)
    assert torch.autograd.gradcheck(lambda a, b, c, d: rua.segment_crf_log_likelihood(a, lens, tags, b, c, d), args)
    z = rua.C(data=x, token_sizes=lens).left(0)
    assert torch.autograd.gradcheck(lambda a, b: z._replace(data=a).crf_log_partition(b),
                                    (z.data.detach().requires_grad_(True), args[1]))


def test_double_backward_raises():
    lens, x, W, st, en, tags = make([3, 2], 4, torch.float64, seed=16)
    xs = x.detach().requires_grad_(True)
    (gx,) = torch.autograd.grad(rua.segment_crf_log_partition(xs, lens, W).sum(), xs, create_graph=True)
    with pytest.raises(RuntimeError):
        gx.sum().backward()


def test_state_kept_only_for_gradients():
    """without a wanted gradient the forward keeps no per-step state (no autograd node at all)"""
    lens, x, W, st, en, tags = make([30, 20], 8, torch.float32, seed=17)
    assert rua.segment_crf_log_partition(x, lens, W).grad_fn is None
    out = rua.segment_crf_log_partition(x, lens, W.detach().requires_grad_(True))
    assert out.grad_fn is not None
