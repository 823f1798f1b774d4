"""CPU-only checks of the SSD (Mamba-2) scan boundary: argument validation happens before any CUDA call, the documented
workspace formula and its monotonicity, and the Python entry points reject bad dtypes, shapes, sizes and CPU tensors
before device work."""
import ctypes
import math

import pytest
import torch


@pytest.fixture(scope='module')
def lib():
    import __graft_entry__ as entry
    entry.build_cuda()
    from torchrua_b200 import _lib
    return _lib.load()


def _structs(layout=0, rows=4, width=0, B=2, off=True, pack=False, srt=True, len_xform=0, Tp=4):
    from torchrua_b200 import _lib
    fake = 0x1000   # never dereferenced: every call below fails validation first
    rg = _lib.Ragged(B, fake if off else None, fake if pack else None, fake if (pack or srt) else None,
                     fake if pack else None, Tp)
    return rg, _lib.Side(layout, len_xform, 0, width, rows)


BAD_LAYOUTS = (dict(rows=-1), dict(B=-1), dict(off=False), dict(srt=False), dict(layout=2, srt=False),
               dict(layout=1, rows=5, width=3), dict(layout=3, rows=5, width=3), dict(layout=9))


def test_ssd_forward_validates_before_cuda(lib):
    fwd, ref = lib.rua_ssd_forward, ctypes.byref
    rg, side = _structs()
    x, dl, A, Bm, Cm, y = (0x1000 * k for k in range(1, 7))

    def call(x=x, dl=dl, A=A, Bm=Bm, Cm=Cm, y=y, H=8, P=4, G=2, N=4, dtype=0, reverse=0, rg=rg, side=side):
        return fwd(x, dl, A, Bm, Cm, None, y, None, H, P, G, N, dtype, reverse, None if rg is None else ref(rg),
                   None if side is None else ref(side), None, 0, None)

    assert call(rg=None) == -1 and call(side=None) == -1
    for dtype in (-1, 4, 7):
        assert call(dtype=dtype) == -1
    assert call(N=0) == -1 and call(P=0) == -1 and call(G=0) == -1 and call(P=-3) == -1
    assert call(G=3) == -1 and call(H=6, G=4) == -1   # H % G != 0
    assert call(P=65) == -3 and call(N=129) == -3 and call(P=128, N=256) == -3
    assert call(H=-1) == -1 and call(reverse=2) == -1 and call(reverse=-1) == -1
    for kw in BAD_LAYOUTS:
        rg2, side2 = _structs(**kw)
        assert call(rg=rg2, side=side2) == -1, kw
    rg3, side3 = _structs(len_xform=1)
    assert call(rg=rg3, side=side3) == -3
    for kw in (dict(x=None), dict(dl=None), dict(A=None), dict(Bm=None), dict(Cm=None), dict(y=None)):
        assert call(**kw) == -1, kw
    # nothing to do: OK without touching anything
    rg4, side4 = _structs(B=0, rows=0)
    assert fwd(None, None, None, None, None, None, None, None, 8, 4, 2, 4, 0, 0, ref(rg4), ref(side4), None, 0,
               None) == 0
    assert call(H=0) == 0


def test_ssd_backward_validates_before_cuda(lib):
    bwd, ref = lib.rua_ssd_backward, ctypes.byref
    rg, side = _structs()
    g, x, dl, A, Bm, Cm, gx, ga = (0x1000 * k for k in range(1, 9))
    need = lib.rua_ssd_workspace_bytes(4, 2, 4, 8, 4, 2, 4, 0)

    def call(g=g, x=x, dl=dl, A=A, Bm=Bm, Cm=Cm, gx=gx, ga=None, H=8, P=4, G=2, N=4, dtype=0, reverse=0, rg=rg,
             side=side, ws=0x9000, nbytes=need):
        return bwd(g, x, dl, A, Bm, Cm, None, gx, None, ga, None, None, None, H, P, G, N, dtype, reverse,
                   None if rg is None else ref(rg), None if side is None else ref(side), ws, nbytes, None)

    assert call(rg=None) == -1 and call(side=None) == -1
    assert call(dtype=5) == -1 and call(N=0) == -1 and call(P=0) == -1 and call(reverse=3) == -1
    assert call(G=3) == -1 and call(P=65) == -3 and call(N=129) == -3
    for kw in BAD_LAYOUTS:
        rg2, side2 = _structs(**kw)
        assert call(rg=rg2, side=side2) == -1, kw
    rg3, side3 = _structs(len_xform=2)
    assert call(rg=rg3, side=side3) == -3
    # the inputs a wanted gradient needs
    for kw in (dict(g=None), dict(x=None), dict(dl=None), dict(A=None), dict(Bm=None), dict(Cm=None)):
        assert call(**kw) == -1, kw
    # every gradient needs the workspace (the backward recomputes the chunk-start states there)
    assert need > 0
    assert call(ws=None) == -2 and call(nbytes=need - 1) == -2 and call(ga=ga, ws=None) == -2
    # nothing wanted: OK
    assert call(gx=None) == 0
    # no sequence and no row: OK without touching anything
    rg4, side4 = _structs(B=0, rows=0)
    assert call(rg=rg4, side=side4, ws=None, nbytes=0) == 0
    assert call(H=0, ws=None, nbytes=0) == 0


@pytest.mark.parametrize('dtype', range(4))
def test_ssd_workspace_formula_and_monotone(lib, dtype):
    ws = lib.rua_ssd_workspace_bytes
    for bad in ((-1, 2, 4, 8, 4, 2, 4, dtype), (8, -1, 4, 8, 4, 2, 4, dtype), (8, 2, -1, 8, 4, 2, 4, dtype),
                (8, 2, 4, -1, 4, 2, 4, dtype), (8, 2, 4, 8, 0, 2, 4, dtype), (8, 2, 4, 8, 65, 2, 4, dtype),
                (8, 2, 4, 8, 4, 0, 4, dtype), (8, 2, 4, 8, 4, 3, 4, dtype), (8, 2, 4, 8, 4, 2, 0, dtype),
                (8, 2, 4, 8, 4, 2, 129, dtype), (8, 2, 4, 8, 4, 2, 4, 4), (8, 2, 4, 8, 4, 2, 4, -1)):
        assert ws(*bad) == 0, bad
    assert ws(0, 2, 4, 8, 4, 2, 4, dtype) == 0 and ws(8, 0, 4, 8, 4, 2, 4, dtype) == 0
    assert ws(8, 2, 4, 0, 4, 2, 4, dtype) == 0
    acc = 8 if dtype == 1 else 4
    Q = 16 if dtype == 1 else 64

    def formula(rows, B, T, H, P, G, N):
        grid = min(B * G, 296)
        return (grid * H * acc + 255) // 256 * 256 + grid * (math.ceil(T / Q) * P * N + T * 2 * N) * acc

    base = dict(rows=4096, B=16, T=1000, H=16, P=64, G=2, N=64)
    steps = dict(rows=(1, 100, 4096, 10 ** 6), B=(1, 7, 16, 40, 1000), T=(0, 1, 63, 64, 65, 4096),
                 H=(2, 4, 16, 64, 256), P=(1, 7, 16, 63, 64), G=(1, 2), N=(1, 5, 64, 65, 128))
    for key, values in steps.items():
        got = []
        for v in values:
            args = dict(base, **{key: v})
            w = ws(args['rows'], args['B'], args['T'], args['H'], args['P'], args['G'], args['N'], dtype)
            assert w == formula(*args.values()), args
            got.append(w)
        assert got == sorted(got), (key, got)
    # G runs over the divisors of H
    got = [ws(4096, 16, 1000, 24, 64, G, 64, dtype) for G in (1, 2, 3, 4, 6, 8, 12, 24)]
    assert got == sorted(got)
    # about 1.8 GB at cfg3 (H = 64, P = 64, N = 128, G = 8, Tmax = 4096, 296 CTAs) for fp32 accumulators
    if acc == 4:
        assert 1.5e9 < ws(10 ** 6, 1000, 4096, 64, 64, 8, 128, dtype) < 2.0e9


def test_ssd_python_rejects_bad_arguments():
    import torchrua_b200 as rua
    lens = torch.tensor([2, 3])
    x, d = torch.randn(5, 4, 3), torch.rand(5, 4)
    A, Bm, Cm = -torch.rand(4), torch.randn(5, 2, 6), torch.randn(5, 2, 6)
    # CPU tensors
    for call in (lambda: rua.segment_ssd(x, lens, d, A, Bm, Cm),
                 lambda: rua.C(data=x, token_sizes=lens).ssd(d, A, Bm, Cm),
                 lambda: rua.L(data=torch.randn(2, 3, 4, 3), token_sizes=lens).ssd(
                     torch.rand(2, 3, 4), A, torch.randn(2, 3, 2, 6), torch.randn(2, 3, 2, 6))):
        with pytest.raises(RuntimeError, match='CUDA tensors only'):
            call()
    # integer payloads, mismatched dtypes
    with pytest.raises(RuntimeError, match='float16/bfloat16/float32/float64'):
        rua.segment_ssd(x.long(), lens, d.long(), A, Bm, Cm)
    with pytest.raises(RuntimeError, match='delta must have dtype'):
        rua.segment_ssd(x, lens, d.double(), A, Bm, Cm)
    with pytest.raises(RuntimeError, match='B must have dtype'):
        rua.segment_ssd(x, lens, d, A, Bm.half(), Cm)
    with pytest.raises(RuntimeError, match='C must have dtype'):
        rua.segment_ssd(x, lens, d, A, Bm, Cm.double())
    with pytest.raises(RuntimeError, match='A must have dtype'):   # A is fp32 for a bf16 payload
        rua.segment_ssd(x.bfloat16(), lens, d.bfloat16(), A.bfloat16(), Bm.bfloat16(), Cm.bfloat16())
    with pytest.raises(RuntimeError, match='initial must have dtype'):
        rua.segment_ssd(x, lens, d, A, Bm, Cm, torch.zeros(2, 4, 3, 6, dtype=torch.float64))
    # shapes
    for bad in (torch.randn(5, 12), torch.randn(5, 4, 3, 1)):
        with pytest.raises(ValueError, match=r'input must be 1 row dimension\(s\) \+ \(H, P\)'):
            rua.segment_ssd(bad, lens, d, A, Bm, Cm)
    for dd in (d[:, :3], d[:4], torch.rand(5, 4, 3)):
        with pytest.raises(ValueError, match='delta must be'):
            rua.segment_ssd(x, lens, dd, A, Bm, Cm)
    for b in (torch.randn(4, 2, 6), torch.randn(5, 12), torch.randn(5, 2, 6, 1)):
        with pytest.raises(ValueError, match='B must be'):
            rua.segment_ssd(x, lens, d, A, b, Cm)
    with pytest.raises(ValueError, match='C must have the shape of B'):
        rua.segment_ssd(x, lens, d, A, Bm, torch.randn(5, 2, 5))
    with pytest.raises(ValueError, match='split into G = 3 groups'):
        rua.segment_ssd(x, lens, d, A, torch.randn(5, 3, 6), torch.randn(5, 3, 6))
    for a in (torch.randn(3), torch.randn(4, 6), torch.randn(1)):
        with pytest.raises(ValueError, match=r'A must be \(H,\)'):
            rua.segment_ssd(x, lens, d, a, Bm, Cm)
    for h0 in (torch.zeros(3, 4, 3, 6), torch.zeros(2, 4, 6, 3), torch.zeros(2, 4, 3)):
        with pytest.raises(ValueError, match='initial must be'):
            rua.segment_ssd(x, lens, d, A, Bm, Cm, h0)
    # head dims outside [1, 64], state sizes outside [1, 128]
    for P in (0, 65):
        with pytest.raises(ValueError, match='head dims 1..64'):
            rua.segment_ssd(torch.randn(5, 4, P), lens, d, A, Bm, Cm)
    for N in (0, 129):
        with pytest.raises(ValueError, match='state sizes 1..128'):
            rua.segment_ssd(x, lens, d, A, torch.randn(5, 2, N), torch.randn(5, 2, N))
    with pytest.raises(ValueError, match='B must be'):
        rua.L(data=torch.randn(2, 3, 4, 3), token_sizes=lens).ssd(torch.rand(2, 3, 4), A, Bm, Cm)


def test_ssd_names_are_exported():
    import torchrua
    import torchrua.ssd
    import torchrua_b200 as rua
    assert torchrua.segment_ssd is rua.segment_ssd
    assert torchrua.ssd.segment_ssd is rua.segment_ssd
    for cls in (rua.C, rua.L, rua.P, rua.R):
        assert callable(cls.ssd)
