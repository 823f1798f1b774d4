"""Prefix scans and the linear recurrence, forward and backward, on every instance of segscan_kernel (csrc/scan.cu): four
dtypes x two vector widths x eight operators = 64 instances, each at 1, 8 and 32 threads across a row, with several column
blocks and with sequences that cross chunk boundaries.  tests/scan_plan.py (pinned on the CPU by test_scan_plan.py) names
the plan of every case.

Every reference is computed in fp64 on the same GPU with plain torch ops (the linear recurrence looped over T), in C
order, once per case and direction, and every layout is compared with it.  Each output is checked two ways:
- formula on the kernel's own saved tensors: cumsum's gradient is the suffix sum of g; logcumsumexp's
  grad_k = sum_{j >= k} g_j exp(x_k - y_j) with the stored y, exactly 0 where x = -inf; cummax / cummin scatter g to the
  kernel's indices (values and indices bit-exact against torch, a gradient only where idx_t == t); the recurrence has
  grad_x = g~ (the adjoint), grad_gate = g~_t y_{t-1} with the stored y (h0 / 0 at the first position) and
  grad_initial = a_0 g~_0 (0 for an empty sequence);
- the true fp64 gradient of the fp64 forward, allowing also for the rounding of the stored output.
The bound is |err| <= e_s(ref) + SLACK u d s: e_s one storage ulp (16-bit) or u_s |ref|, u the accumulator's unit
roundoff, s the same computation on absolute values, d the depth of the kernel's combination tree from the plan.  Rows that
hold no token pass through (grad_gate 0), C and P give the same bits, and the wide cases give the same bits run to run."""
import math
import re

import numpy as np
import pytest
import torch

import torchrua_b200 as rua
from tests import scan_plan
from tests.test_gpu_scan import oracle as torch_scan

pytestmark = pytest.mark.gpu

DEV = torch.device('cuda')
F64, F32, F16, BF16 = torch.float64, torch.float32, torch.float16, torch.bfloat16
DTYPES = [F32, F64, F16, BF16]
LAYOUTS = ['C', 'L', 'P', 'R']
FAMILIES = ['sum', 'logsumexp', 'max', 'min', 'linrec']
KINDS = dict(scan_plan.SCAN_KINDS, linrec=('linrec', 'linrec_bwd'))
FREE = {'sum': rua.segment_cumsum, 'logsumexp': rua.segment_logcumsumexp, 'max': rua.segment_cummax,
        'min': rua.segment_cummin}
METHOD = {'sum': 'cumsum', 'logsumexp': 'logcumsumexp', 'max': 'cummax', 'min': 'cummin'}

# unit roundoff of the accumulator (fp32 for 16-bit payloads) and of fp32 / fp64 storage
U_ACC = {F64: 2.0 ** -53, F32: 2.0 ** -24, F16: 2.0 ** -24, BF16: 2.0 ** -24}
# explicit mantissa bits and smallest normal exponent of the 16-bit formats: one storage ulp
MANT = {F16: 10, BF16: 7}
EMIN = {F16: -14, BF16: -126}
# error per level of the combination tree, in units of u times the absolute computation: one rounding for a sum, a
# product and an fma for the affine maps, exp + fma for the logcumsumexp backward, and for logaddexp exp, log1p and an add
# (the fast fp32 intrinsics of the 16-bit instances stay within 8 u absolute there)
SLACK = 16
EXTRA_W = 3   # L / R storage wider than the longest sequence: padding rows land inside chunks

# regime -> H as a function of the vector width VV (elements per 16 bytes), and the (V == VV, tpc, ncb) its forward plan has
REGIMES = {'narrow-1': (lambda VV: 1, (False, 1, 1)), 'narrow-vec': (lambda VV: VV, (True, 1, 1)),
           'mid-vec': (lambda VV: 8 * VV, (True, 8, 1)), 'mid-odd': (lambda VV: 7, (False, 8, 1)),
           'wide-vec': (lambda VV: 75 * VV, (True, 32, 3)), 'wide-odd': (lambda VV: 301, (False, 32, 10)),
           'misaligned': (lambda VV: 75 * VV, (False, 32, None))}


def _dn(dtype):
    return {F64: 'f64', F32: 'f32', F16: 'f16', BF16: 'bf16'}[dtype]


def aligned(regime, kind, backward):
    """the misaligned regime shifts the payload (scans) or the initial state (recurrence) one element off 16 bytes; the
    backward of cumsum and cummax / cummin reads only grad_out and the indices, which are aligned"""
    return regime != 'misaligned' or (backward and kind in ('sum', 'run_bwd'))


def plans(dtype, regime, family, rows=1):
    H = REGIMES[regime][0](scan_plan.vec_width(dtype))
    kf, kb = KINDS[family]
    return (scan_plan.plan(kf, rows, H, dtype, aligned(regime, kf, False)),
            scan_plan.plan(kb, rows, H, dtype, aligned(regime, kb, True)))


# ---------------------------------------------------------------------------------------------------------------------
# sequences in C order
# ---------------------------------------------------------------------------------------------------------------------
class Seqs:
    """index maps of a batch of sequences in C order: scan order (every sequence reversed for reverse=True) and the
    time-major zero-padded (T, B, H) form"""

    def __init__(self, lens):
        ls = torch.tensor(lens, dtype=torch.long, device=DEV)
        self.lens, self.B, self.n, self.T = ls, len(lens), int(sum(lens)), max(list(lens) + [1])
        self.off = torch.cumsum(ls, 0) - ls
        self.seg = torch.repeat_interleave(torch.arange(self.B, device=DEV), ls)
        self.t = torch.arange(self.n, device=DEV) - self.off[self.seg]
        self.rrows = self.off[self.seg] + ls[self.seg] - 1 - self.t

    def order(self, v, rev):
        """C order <-> scan order (an involution)"""
        return v[self.rrows] if rev else v

    def pad(self, v):
        p = torch.zeros((self.T, self.B) + tuple(v.shape[1:]), dtype=v.dtype, device=DEV)
        p[self.t, self.seg] = v
        return p

    def unpad(self, p):
        return p[self.t, self.seg]

    def scan(self, fn, v, rev):
        """fn along time in scan order, applied to every sequence; C order in and out"""
        return self.order(self.unpad(fn(self.pad(self.order(v, rev)))), rev)

    def cumsum(self, v, rev):
        return self.scan(lambda p: torch.cumsum(p, 0), v, rev)

    def seq_max(self, v):
        """(B, H) maximum of every sequence, -inf for an empty one"""
        out = torch.full((self.B,) + tuple(v.shape[1:]), -float('inf'), dtype=v.dtype, device=DEV)
        return out.scatter_reduce(0, self.seg.view(-1, 1).expand_as(v), v, 'amax')

    def spans(self, pos, R):
        """chunks of R virtual positions every sequence's positions touch"""
        ch = pos // R
        lo = torch.full((self.B,), 1 << 62, dtype=torch.long, device=DEV).scatter_reduce(0, self.seg, ch, 'amin')
        hi = torch.full((self.B,), -1, dtype=torch.long, device=DEV).scatter_reduce(0, self.seg, ch, 'amax')
        return (hi - lo + 1).clamp(min=0)


def case_lengths(Rs, seed):
    """lengths (C order, unsorted) for plans with rows per chunk Rs: an empty and a 1-row sequence at the start, two long
    sequences over >= 3 chunks of the larger R, short ones (<= 64 rows), and for every R an empty and a 1-row sequence on a
    boundary, a sequence of exactly R rows from one boundary to the next, one that ends one row before a boundary, a 1-row
    sequence on the last row before it and one on the boundary, and one that starts one row after it.  The total is a
    multiple of every R, so the boundaries of reverse=True (counted from the end) are the same rows."""
    rng = np.random.default_rng(seed)
    L, M = max(Rs), math.lcm(*Rs)
    lens, marks = [], {}

    def add(n):
        lens.append(int(n))
        return len(lens) - 1

    def fill_to(mult, rem):
        while (rem - sum(lens)) % mult:
            add(min((rem - sum(lens)) % mult, int(rng.integers(1, max(2, L // 3)))))

    add(0)
    add(1)
    marks['long1'] = add(3 * L + 7)
    marks['short'] = [add(n) for n in rng.integers(2, 65, 6)]
    for R in sorted(set(Rs)):
        fill_to(R, 0)
        add(0)
        add(1)
        fill_to(R, 0)
        marks.setdefault('exact', add(R))
        n = R // 2 + 3
        fill_to(R, -(n + 1))
        add(n)
        add(1)
        add(1)
        add(n)
    marks['long2'] = add(3 * L + 5)
    fill_to(M, 0)
    return lens, marks, M


# ---------------------------------------------------------------------------------------------------------------------
# error model
# ---------------------------------------------------------------------------------------------------------------------
def e_store(ref, dtype):
    """the storage rounding allowed at ref: one ulp for 16-bit (faithful rounding), u_s |ref| for fp32 / fp64"""
    if dtype in (F32, F64):
        return U_ACC[dtype] * ref.abs()
    _, e = torch.frexp(ref)
    e = torch.where(ref == 0, torch.full_like(e, EMIN[dtype]), (e - 1).clamp(min=EMIN[dtype]))
    return torch.ldexp(torch.ones_like(ref), e - MANT[dtype])


def check(what, got, ref, bound):
    """|got - ref| <= bound where ref is finite; infinite references are matched exactly"""
    got = got.double()
    fin = torch.isfinite(ref)
    ok = torch.where(fin, (got - ref).abs() <= bound, got == ref)
    if not bool(ok.all()):
        bad = (~ok).nonzero()
        k = tuple(bad[0].tolist())
        raise AssertionError(f'{what}: {bad.shape[0]} elements out of bounds, first at {k}: got {got[k].item()!r}, '
                             f'ref {ref[k].item()!r}, bound {bound[k].item() if torch.is_tensor(bound) else bound!r}')


def bits(t):
    return t.contiguous().view({8: torch.int64, 4: torch.int32, 2: torch.int16}[t.element_size()])


# ---------------------------------------------------------------------------------------------------------------------
# references (fp64, C order)
# ---------------------------------------------------------------------------------------------------------------------
def linrec_loop(x, a, h0, g, seqs, rev):
    """h_t = a_t h_{t-1} + x_t in scan order and its adjoint g~_t = g_t + a_{t+1} g~_{t+1} written out as a reverse loop,
    each with its absolute-value companion (|a|, |x|, |h0|, |g|)"""
    px, pa, pg = (seqs.pad(seqs.order(v, rev)) for v in (x, a, g))
    A, X, G = (torch.stack([p, p.abs()], 1) for p in (pa, px, pg))
    init = torch.zeros_like(px[0]) if h0 is None else h0
    h = torch.stack([init, init.abs()])
    hs = []
    for k in range(seqs.T):
        h = torch.addcmul(X[k], A[k], h)
        hs.append(h)
    Y = torch.stack(hs)
    A1 = torch.cat([A[1:], torch.zeros_like(A[:1])])   # a_{t+1}; 0 past the end of every sequence
    gt = torch.zeros_like(h)
    gts = [None] * seqs.T
    for k in reversed(range(seqs.T)):
        gt = torch.addcmul(G[k], A1[k], gt)
        gts[k] = gt
    GT = torch.stack(gts)
    un = lambda p: seqs.order(seqs.unpad(p), rev)   # noqa: E731
    yprev = torch.cat([init[None], Y[:-1, 0]])
    return dict(y=un(Y[:, 0]), s_y=un(Y[:, 1]), gt=un(GT[:, 0]), s_gt=un(GT[:, 1]), yprev=un(yprev),
                gh=pa[0] * GT[0, 0], s_gh=pa[0].abs() * GT[0, 1])


def prev_in_scan(y, h0, seqs, rev):
    """y at the previous position of the same sequence in scan order, h0 (or 0) at the first"""
    p = seqs.pad(seqs.order(y, rev))
    init = torch.zeros_like(p[0]) if h0 is None else h0
    return seqs.order(seqs.unpad(torch.cat([init[None], p[:-1]])), rev)


def lse_grad(x, y, g, seqs, rev, weight=None):
    """sum_{j >= k} g_j exp(x_k - y_j) over the rest of the sequence in scan order (0 where x = -inf), with a
    per-sequence shift; weight multiplies every term j (the absolute and rounding companions)"""
    fin = torch.isfinite(y)
    c = seqs.seq_max(torch.where(fin, y, -float('inf')))
    c = torch.where(torch.isfinite(c), c, torch.zeros_like(c))[seqs.seg]
    w = torch.where(fin, g * torch.exp(c - torch.where(fin, y, c)), torch.zeros_like(g))
    if weight is not None:
        w = w * torch.where(fin, weight, torch.zeros_like(weight))
    return torch.where(x == -float('inf'), torch.zeros_like(x), torch.exp(x - c) * seqs.cumsum(w, not rev))


def run_grad(g, idx, seqs):
    """g scattered to the position each row's index names (cummax / cummin backward)"""
    n, H = g.shape
    tgt = (seqs.off[seqs.seg].view(-1, 1) + idx) * H + torch.arange(H, device=DEV)
    return torch.zeros(n * H, dtype=F64, device=DEV).index_add_(0, tgt.flatten(), g.flatten()).view(n, H)


# ---------------------------------------------------------------------------------------------------------------------
# one case: dtype x regime x op family
# ---------------------------------------------------------------------------------------------------------------------
class Case:
    def __init__(self, dtype, regime, family, seed):
        self.dtype, self.regime, self.family = dtype, regime, family
        self.H = H = REGIMES[regime][0](scan_plan.vec_width(dtype))
        self.kf, self.kb = KINDS[family]
        pf, pb = plans(dtype, regime, family)
        lens, self.marks, M = case_lengths(sorted({pf.R, pb.R}), seed)
        self.lens, self.seqs = lens, Seqs(lens)
        self.tail = M                     # C rows past sum(sizes): whole chunks, so C and P chunk alike both ways
        self.W = max(lens) + EXTRA_W
        self.lens_t = self.seqs.lens
        self.sum_loss = regime == 'mid-odd'   # grad_out from y.sum(): a stride-0 cotangent
        n, B = self.seqs.n, len(lens)
        gen = torch.Generator(device=DEV).manual_seed(seed)
        rnd = lambda *s: torch.rand(s, generator=gen, device=DEV, dtype=F64)     # noqa: E731
        nrm = lambda *s: torch.randn(s, generator=gen, device=DEV, dtype=F64)    # noqa: E731
        signed = lambda *s: torch.where(rnd(*s) < 0.5, -1.0, 1.0) * (0.5 + 1.5 * rnd(*s))   # noqa: E731
        off = self.seqs.off.tolist()
        o1, n1 = off[self.marks['long1']], lens[self.marks['long1']]
        o2, n2 = off[self.marks['long2']], lens[self.marks['long2']]
        rmin = min(pf.R, pb.R)
        rows = max(B * self.W, n + self.tail)
        if family == 'sum':
            x = nrm(n, H)
        elif family == 'logsumexp':
            x = 3 * nrm(n, H)
            x[rnd(n, H) < 0.03] = -float('inf')
            x[o1:o1 + rmin + 5] = -float('inf')           # leads long1 across a chunk boundary (forward)
            x[o2 + n2 - rmin - 5:o2 + n2] = -float('inf')  # leads long2 across a boundary (reverse)
            oe = off[self.marks['exact']]
            x[oe:oe + lens[self.marks['exact']]] = -float('inf')   # a whole sequence of -inf
        elif family in ('max', 'min'):
            x = torch.randint(-3, 4, (n, H), generator=gen, device=DEV).double()
            x[o1 + 1] = x[o1 + n1 - 2] = 10.0             # an early maximum owns a run over many chunks (both ways)
            x[o1 + 2] = x[o1 + n1 - 3] = -10.0
            x[o2 + n2 // 2] = float('nan')                # a NaN sticks from the middle of long2
        else:
            x = nrm(n, H)
            kind = torch.tensor([i % 2 for i in range(B)], device=DEV)[self.seqs.seg].view(-1, 1)
            a = torch.where(kind == 0, rnd(n, H), 2 * rnd(n, H) - 1)       # [0, 1) or signed |a| <= 1
            for i in self.marks['short']:                                   # |a| up to 1.1 in short sequences only
                a[off[i]:off[i] + lens[i]] = 2.2 * rnd(lens[i], H) - 1.1
            a[rnd(n, H) < 0.05] = 0.0
            for R in {pf.R, pb.R}:
                a[0:n:2 * R] = 0.0                                          # resets on chunk boundaries
            q = rmin // 4
            a[o2 + 10:o2 + 10 + 2 * q] = 1.0                                # runs of exactly +1 and -1
            a[o2 + 10 + 2 * q:o2 + 10 + 3 * q] = -1.0
            self.a = a.to(dtype)
            self.h0 = nrm(B, H).to(dtype)
            self.a_noise = nrm(rows, H).to(dtype)
        self.x = x.to(dtype)
        self.g = torch.ones(n, H, dtype=dtype, device=DEV) if self.sum_loss else signed(n, H).to(dtype)
        self.x_noise = (7 * nrm(rows, H)).to(dtype)
        self.g_noise = torch.ones(rows, H, dtype=dtype, device=DEV) if self.sum_loss else signed(rows, H).to(dtype)
        tmpl = rua.C(data=torch.zeros(n, H, dtype=dtype, device=DEV), token_sizes=self.lens_t)
        self.tmpl = {'P': tmpl.pack(), 'L': tmpl.left(0), 'R': tmpl.right(0)}
        pidx = rua.C(data=torch.arange(n, dtype=F64, device=DEV).view(-1, 1), token_sizes=self.lens_t).pack().data
        self.p_rows = torch.empty(n, dtype=torch.long, device=DEV)
        self.p_rows[pidx[:, 0].long()] = torch.arange(n, device=DEV)

    # ---- storage of each layout ------------------------------------------------------------------------------------
    def layout_rows(self, layout):
        """(storage rows, storage row of every C-order token, virtual position of every token)"""
        s, n = self.seqs, self.seqs.n
        if layout == 'C':
            return n + self.tail, torch.arange(n, device=DEV), torch.arange(n, device=DEV)
        if layout == 'P':
            return n, self.p_rows, torch.arange(n, device=DEV)
        lead = 0 if layout == 'L' else self.W - s.lens[s.seg]
        pos = s.seg * self.W + lead + s.t
        return len(self.lens) * self.W, pos, pos

    def storage(self, layout, v, noise):
        rows, tok, _ = self.layout_rows(layout)
        st = noise[:rows].clone()
        st[tok] = v
        return st

    def depth(self, layout, rev, p):
        """per token: the height of the kernel's combination tree -- kRG rows of a group, log2(G) Kogge-Stone levels, one
        compose per chunk the sequence spans, kRG replayed rows in pass 2, + 2"""
        rows, _, pos = self.layout_rows(layout)
        if rev:
            pos = rows - 1 - pos
        spans = self.seqs.spans(pos, p.R)
        return (2 * (p.R // p.G) + (p.G.bit_length() - 1) + spans + 2)[self.seqs.seg].view(-1, 1).double()

    def variant(self, layout, rev):
        """linear recurrence: (initial given, x frozen, gate frozen); C and P share theirs so their bits compare"""
        cp = layout in ('C', 'P')
        init = self.regime == 'misaligned' or cp != rev
        return init, (not cp and not rev), (cp and rev)

    # ---- one layout, one direction ----------------------------------------------------------------------------------
    def run(self, layout, rev):
        """kernel results in C order (y, idx, gx, gg, gh); non-token rows checked to pass through"""
        H, n = self.H, self.seqs.n
        rows, tok, _ = self.layout_rows(layout)
        nt = torch.ones(rows, dtype=torch.bool, device=DEV)
        nt[tok] = False
        mis = self.regime == 'misaligned'
        shape = (len(self.lens), self.W, H) if layout in ('L', 'R') else (rows, H)
        z = self.tmpl.get(layout)
        xs = self.storage(layout, self.x, self.x_noise)
        gs = self.storage(layout, self.g, self.g_noise)
        if self.family == 'linrec':
            init, fx, fg = self.variant(layout, rev)
            xl = xs.clone().requires_grad_(not fx)
            al = self.storage(layout, self.a, self.a_noise).requires_grad_(not fg)
            hl = self.h0.clone().requires_grad_(True) if init else None
            hin = shifted(hl) if (init and mis) else hl
            if layout == 'C':
                y = rua.segment_linear_recurrence(xl, self.lens_t, al, hin, reverse=rev)
            else:
                y = z._replace(data=xl.view(shape)).linear_recurrence(al.view(shape), hin, reverse=rev).data
            y = y.reshape(rows, H)
            leaves = [t for t in (xl, al, hl) if t is not None and t.requires_grad]
            outs, idx = y, None
        else:
            xl = xs.clone().requires_grad_(True)
            xin = shifted(xl) if mis else xl
            if layout == 'C':
                res = FREE[self.family](xin, self.lens_t, reverse=rev)
                outs, idx = (res.values, res.indices) if self.family in ('max', 'min') else (res, None)
            else:
                res = getattr(z._replace(data=xin.view(shape)), METHOD[self.family])(reverse=rev)
                outs, idx = (res[0].data, res[1].data) if self.family in ('max', 'min') else (res.data, None)
            outs = outs.reshape(rows, H)
            idx = None if idx is None else idx.reshape(rows, H)
            leaves = [xl]
        if self.sum_loss:
            grads = torch.autograd.grad(outs.sum(), leaves)
        else:
            grads = torch.autograd.grad(outs, leaves, gs)
        grads = list(grads)
        r = dict(y=outs.detach()[tok])
        # rows that hold no token: copied through (index 0), grad_out passed through, gate gradient 0
        assert torch.equal(bits(outs.detach()[nt]), bits(xs[nt])), 'non-token rows not copied through'
        if idx is not None:
            r['idx'] = idx[tok]
            assert (idx[nt] == 0).all()
        if self.family == 'linrec':
            for name, leaf in (('gx', xl), ('gg', al), ('gh', hl)):
                if leaf is not None and leaf.requires_grad:
                    gr = grads.pop(0)
                    r[name] = gr if name == 'gh' else gr[tok]
                    if name == 'gx':
                        assert torch.equal(bits(gr[nt]), bits(gs[nt])), 'grad_x of non-token rows is not grad_out'
                    if name == 'gg':
                        assert (gr[nt] == 0).all(), 'grad_gate of non-token rows is not 0'
        else:
            r['gx'] = grads[0][tok]
            assert torch.equal(bits(grads[0][nt]), bits(gs[nt])), 'gradient of non-token rows is not grad_out'
        return r

    # ---- the references of one direction ----------------------------------------------------------------------------
    def refs(self, rev):
        s, x, g = self.seqs, self.x.double(), self.g.double()
        f = self.family
        if f == 'sum':
            return dict(y=s.cumsum(x, rev), s_y=s.cumsum(x.abs(), rev), gx=s.cumsum(g, not rev),
                        s_gx=s.cumsum(g.abs(), not rev))
        if f == 'logsumexp':
            y = s.scan(lambda p: torch.logcumsumexp(p, 0), x, rev)
            return dict(y=y, s_y=y.abs() + 1)
        if f in ('max', 'min'):
            v, i = torch_scan(f, self.x, self.lens, rev)
            return dict(y=v, idx=i, gx=run_grad(g, i, s), s_gx=run_grad(g.abs(), i, s))
        h0 = self.h0.double()
        return dict(init=linrec_loop(x, self.a.double(), h0, g, s, rev),
                    zero=linrec_loop(x, self.a.double(), None, g, s, rev))

    def check(self, r, ref, layout, rev):
        dt, u = self.dtype, U_ACC[self.dtype]
        s, x, g = self.seqs, self.x.double(), self.g.double()
        pf, pb = plans(dt, self.regime, self.family)
        d_f, d_b = self.depth(layout, rev, pf), self.depth(layout, rev, pb)
        tag = f'{layout} reverse={rev}'
        f = self.family
        if f in ('max', 'min'):
            assert torch.equal(torch.isnan(r['y']), torch.isnan(ref['y'])), f'{tag}: NaN positions'
            assert torch.equal(r['y'].nan_to_num(0.0), ref['y'].nan_to_num(0.0)), f'{tag}: values'
            assert torch.equal(r['idx'], ref['idx']), f'{tag}: indices'
            gx = r['gx'].double()
            check(f'{tag} grad', gx, ref['gx'], e_store(ref['gx'], dt) + SLACK * u * d_b * ref['s_gx'])
            assert ((gx == 0) | (r['idx'] == s.t.view(-1, 1))).all(), f'{tag}: gradient off a run start'
            return
        if f == 'sum':
            check(f'{tag} y', r['y'], ref['y'], e_store(ref['y'], dt) + SLACK * u * d_f * ref['s_y'])
            check(f'{tag} grad', r['gx'], ref['gx'], e_store(ref['gx'], dt) + SLACK * u * d_b * ref['s_gx'])
            return
        if f == 'logsumexp':
            check(f'{tag} y', r['y'], ref['y'], e_store(ref['y'], dt) + SLACK * u * d_f * ref['s_y'])
            yh = r['y'].double()
            form = lse_grad(x, yh, g, s, rev)
            sb = lse_grad(x, yh, g.abs(), s, rev)
            check(f'{tag} grad (stored y)', r['gx'], form, e_store(form, dt) + SLACK * u * d_b * sb)
            assert (r['gx'][x == -float('inf')] == 0).all(), f'{tag}: gradient at -inf is not 0'
            # |got - true| <= |got - form| + |form - true|: the kernel rounds a value near form, so the storage ulp is
            # that of form, and |form - true| <= sum_j |g_j| exp(x_k - y_j) expm1|y_j - y^_j|
            true = lse_grad(x, ref['y'], g, s, rev)
            rnd = lse_grad(x, ref['y'], g.abs(), s, rev, torch.expm1((ref['y'] - yh).abs()))
            check(f'{tag} grad (fp64 y)', r['gx'], true, e_store(form, dt) + SLACK * u * d_b * sb + rnd)
            return
        init, fx, fg = self.variant(layout, rev)
        lr = ref['init' if init else 'zero']
        check(f'{tag} y', r['y'], lr['y'], e_store(lr['y'], dt) + SLACK * u * d_f * lr['s_y'])
        if not fx:
            check(f'{tag} grad_x', r['gx'], lr['gt'], e_store(lr['gt'], dt) + SLACK * u * d_b * lr['s_gt'])
        if not fg:
            yprev = prev_in_scan(r['y'].double(), self.h0.double() if init else None, s, rev)
            form = lr['gt'] * yprev
            sb = lr['s_gt'] * yprev.abs()
            check(f'{tag} grad_gate (stored y)', r['gg'], form, e_store(form, dt) + SLACK * u * d_b * sb)
            true = lr['gt'] * lr['yprev']   # as for logcumsumexp: the storage ulp of form, + |g~_t| |y_{t-1} - y^_{t-1}|
            rnd = lr['gt'].abs() * (lr['yprev'] - yprev).abs()
            check(f'{tag} grad_gate (fp64 y)', r['gg'], true, e_store(form, dt) + SLACK * u * d_b * sb + rnd)
        if init:
            # the deepest token of every sequence bounds its grad_initial; an empty sequence gets exactly 0
            dmax = torch.zeros(s.B, 1, dtype=F64, device=DEV).scatter_reduce(0, s.seg.view(-1, 1), d_b, 'amax')
            check(f'{tag} grad_initial', r['gh'], lr['gh'], e_store(lr['gh'], dt) + SLACK * u * dmax * lr['s_gh'])
            empty = s.lens == 0
            assert (r['gh'][empty] == 0).all(), f'{tag}: grad_initial of an empty sequence'


def shifted(t):
    """a copy of t (in the autograd graph) whose data pointer is one element past 16-byte alignment"""
    buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    v = buf[1:].view(t.shape)
    v.copy_(t)
    assert v.data_ptr() % 16 != 0
    return v


CASES = [(dt, rg, fam) for dt in DTYPES for rg in REGIMES for fam in FAMILIES]


def _cid(dt, rg, fam):
    return f'{rg}-{_dn(dt)}-{fam}'


@pytest.mark.parametrize('dtype,regime,family', CASES, ids=[_cid(*c) for c in CASES])
def test_case(dtype, regime, family):
    """every layout and direction against the fp64 references; C and P bit-identical; the wide cases deterministic"""
    case = Case(dtype, regime, family, seed=CASES.index((dtype, regime, family)))
    pf, pb = plans(dtype, regime, family, rows=case.seqs.n)
    want_vec, tpc, ncb = REGIMES[regime][1]
    assert (pf.V > 1, pf.tpc) == (want_vec, tpc) and ncb in (None, pf.ncb), pf
    if regime.startswith('wide') or regime == 'misaligned':
        assert pf.ncb >= 3 and pb.ncb >= 3
        pos = torch.arange(case.seqs.n, device=DEV)
        for p in (pf, pb):
            assert int(case.seqs.spans(pos, p.R)[case.marks['long1']]) >= 3
    first = {}
    for rev in (False, True):
        ref = case.refs(rev)
        got = {}
        for layout in LAYOUTS:
            got[layout] = case.run(layout, rev)
            case.check(got[layout], ref, layout, rev)
        # C and P share the virtual order and the chunks: the same bits
        assert got['C'].keys() == got['P'].keys()
        for k in got['C']:
            assert torch.equal(bits(got['C'][k]), bits(got['P'][k])), f'C and P differ in {k} (reverse={rev})'
        first = first or got['C']
    if regime in ('wide-vec', 'wide-odd'):
        again = case.run('C', False)
        for k in first:
            assert torch.equal(bits(first[k]), bits(again[k])), f'{k} differs run to run'


# ---------------------------------------------------------------------------------------------------------------------
# structural checks
# ---------------------------------------------------------------------------------------------------------------------
_KERNEL = re.compile(r'segscan_kernel<(.*)>\s*\(')


def _norm(name):
    m = _KERNEL.search(name)
    if not m:
        return None
    inner = m.group(1).replace('rua::', '').replace('(anonymous namespace)::', '').replace(' ', '')
    return f'segscan_kernel<{inner}>'


def test_every_case_runs_the_kernel_it_names():
    """under the profiler, each case's forward and backward launch exactly the instance the plan names, one each, in
    order; together the cases run all 64 instances, each at 1, 8 and 32 threads across a row"""
    from torch.profiler import ProfilerActivity, profile
    lens = [5, 0, 3, 1]
    ls = torch.tensor(lens, device=DEV)
    calls, want = [], []
    for dtype, regime, family in CASES:
        H = REGIMES[regime][0](scan_plan.vec_width(dtype))
        mis = regime == 'misaligned'
        x = torch.randn(sum(lens), H, device=DEV).to(dtype)
        a = torch.rand(sum(lens), H, device=DEV).to(dtype)
        h0 = torch.randn(len(lens), H, device=DEV).to(dtype)
        calls.append((family, x, a, h0, mis))
        for backward, kind in enumerate(KINDS[family]):
            p = scan_plan.plan(kind, sum(lens), H, dtype, aligned(regime, kind, bool(backward)))
            want.append((scan_plan.instance(kind, dtype, p.V, family), p.tpc, _cid(dtype, regime, family)))
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for family, x, a, h0, mis in calls:
            xl = x.clone().requires_grad_(True)
            if family == 'linrec':
                hl = h0.clone().requires_grad_(True)
                al = a.clone().requires_grad_(True)
                y = rua.segment_linear_recurrence(xl, ls, al, shifted(hl) if mis else hl)
                torch.autograd.grad(y, (xl, al, hl), torch.ones_like(y))
            else:
                res = FREE[family](shifted(xl) if mis else xl, ls)
                y = res.values if family in ('max', 'min') else res
                torch.autograd.grad(y, xl, torch.ones_like(y))
        torch.cuda.synchronize()
    kernels = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and _norm(e.name)),
                     key=lambda e: e.time_range.start)
    got = [_norm(e.name) for e in kernels]
    assert len(got) == len(want), f'{len(got)} scan kernels launched for {len(want)} calls'
    for g_name, (w_name, _, cid) in zip(got, want):
        assert g_name == w_name, f'{cid}: launched {g_name}, expected {w_name}'
    seen = {}
    for name, tpc, _ in want:
        seen.setdefault(name, set()).add(tpc)
    assert len(seen) == 64
    for name, tpcs in seen.items():
        assert {1, 8, 32} <= tpcs, f'{name} ran at tpc {sorted(tpcs)} only'


def test_linrec_adjoint_matches_autograd():
    """the explicit reverse-loop adjoint of linrec_loop against torch autograd of its forward loop"""
    lens = [5, 0, 9, 1, 4]
    s = Seqs(lens)
    gen = torch.Generator(device=DEV).manual_seed(11)
    x, a, g = (torch.randn(s.n, 3, generator=gen, device=DEV, dtype=F64) for _ in range(3))
    h0 = torch.randn(len(lens), 3, generator=gen, device=DEV, dtype=F64)
    for rev in (False, True):
        for init in (h0, None):
            leaves = [t.clone().requires_grad_(True) for t in (x, a) + ((init,) if init is not None else ())]
            hl = leaves[2] if init is not None else None
            y = linrec_loop(leaves[0], leaves[1], hl, g, s, rev)['y']
            want = torch.autograd.grad(y, leaves, g)
            r = linrec_loop(x, a, init, g, s, rev)
            torch.testing.assert_close(r['gt'], want[0], rtol=1e-12, atol=1e-12)
            torch.testing.assert_close(r['gt'] * r['yprev'], want[1], rtol=1e-12, atol=1e-12)
            if init is not None:
                torch.testing.assert_close(r['gh'], want[2], rtol=1e-12, atol=1e-12)
            torch.testing.assert_close(r['y'], y.detach())


@pytest.mark.parametrize('dtype', DTYPES)
def test_logcumsumexp_gradient_around_plus_inf(dtype):
    """y = +inf from a +inf input on: every later position has gradient exactly 0 (d y_j / d x_k = exp(x_k - inf)), and the
    positions before it get the gradient of the finite prefix alone, across chunk carries on both sides"""
    H = 1
    n = 5000
    gen = torch.Generator(device=DEV).manual_seed(12)
    x = (3 * torch.randn(n, H, generator=gen, device=DEV, dtype=F64)).to(dtype)
    p = 2100
    x[p] = float('inf')
    lens = [n]
    ls = torch.tensor(lens, device=DEV)
    g = (0.5 + torch.rand(n, H, generator=gen, device=DEV, dtype=F64)).to(dtype)
    s = Seqs(lens)
    for rev in (False, True):
        xl = x.clone().requires_grad_(True)
        y = rua.segment_logcumsumexp(xl, ls, reverse=rev)
        (gx,) = torch.autograd.grad(y, xl, g)
        after = torch.arange(n, device=DEV) < p if rev else torch.arange(n, device=DEV) > p
        before = torch.arange(n, device=DEV) > p if rev else torch.arange(n, device=DEV) < p
        assert (gx[after] == 0).all(), f'reverse={rev}: gradient after +inf'
        assert torch.isfinite(gx[before]).all(), f'reverse={rev}: non-finite gradient before +inf'
        yh = y.detach().double()
        form = lse_grad(x.double(), torch.where(before.view(-1, 1), yh, torch.full_like(yh, float('inf'))),
                        g.double(), s, rev)
        sb = lse_grad(x.double(), torch.where(before.view(-1, 1), yh, torch.full_like(yh, float('inf'))),
                      g.double().abs(), s, rev)
        pl = scan_plan.plan('lse_bwd', n, H, dtype)
        d = 2 * (pl.R // pl.G) + (pl.G.bit_length() - 1) + (n // pl.R + 2) + 2
        check(f'reverse={rev} before +inf', gx[before], form[before],
              e_store(form[before], dtype) + SLACK * U_ACC[dtype] * d * sb[before])
