"""CPU-only checks of the selective-scan boundary: argument validation happens before any CUDA call, the documented
state and workspace bounds, and the Python entry points reject bad dtypes, shapes, state sizes and CPU tensors before
device work."""
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


def _structs(layout=0, rows=4, width=0, B=2, off=True, pack=False, srt=True, len_xform=0):
    from torchrua_b200 import _lib
    fake = 0x1000   # never dereferenced: every call below fails validation first
    rg = _lib.Ragged(B, fake if off else None, fake if pack else None, fake if (pack or srt) else None,
                     fake if pack else None, 1 if pack else 0)
    return rg, _lib.Side(layout, len_xform, 0, width, rows)


BAD_LAYOUTS = (dict(rows=-1), dict(B=-1), dict(off=False), dict(srt=False), dict(layout=2, srt=False),
               dict(layout=1, rows=5, width=3), dict(layout=3, rows=5, width=3), dict(layout=9))


def test_ssm_forward_validates_before_cuda(lib):
    fwd, ref = lib.rua_ssm_forward, ctypes.byref
    rg, side = _structs()
    x, dl, A, Bm, Cm, y = (0x1000 * k for k in range(1, 7))

    def call(x=x, dl=dl, A=A, Bm=Bm, Cm=Cm, y=y, H=8, N=4, dtype=0, reverse=0, rg=rg, side=side):
        return fwd(x, dl, A, Bm, Cm, None, y, None, None, H, N, dtype, reverse, None if rg is None else ref(rg),
                   None if side is None else ref(side), None, 0, None)

    assert call(rg=None) == -1 and call(side=None) == -1
    for dtype in (-1, 4, 7):
        assert call(dtype=dtype) == -1
    assert call(N=0) == -1 and call(N=-2) == -1
    assert call(N=17) == -3 and call(N=64) == -3
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
    assert fwd(None, None, None, None, None, None, None, None, None, 8, 4, 0, 0, ref(rg4), ref(side4), None, 0, None) == 0
    assert call(H=0) == 0


def test_ssm_backward_validates_before_cuda(lib):
    bwd, ref = lib.rua_ssm_backward, ctypes.byref
    rg, side = _structs()
    g, x, dl, A, Bm, Cm, st, gx, ga = (0x1000 * k for k in range(1, 10))

    def call(g=g, x=x, dl=dl, A=A, Bm=Bm, Cm=Cm, st=st, gx=gx, ga=None, gb=None, H=8, N=4, dtype=0, reverse=0, rg=rg,
             side=side, ws=None, nbytes=0):
        return bwd(g, x, dl, A, Bm, Cm, st, gx, None, ga, gb, None, None, H, N, dtype, reverse,
                   None if rg is None else ref(rg), None if side is None else ref(side), ws, nbytes, None)

    assert call(rg=None) == -1 and call(side=None) == -1
    assert call(dtype=5) == -1 and call(N=0) == -1 and call(N=17) == -3 and call(reverse=3) == -1
    for kw in BAD_LAYOUTS:
        rg2, side2 = _structs(**kw)
        assert call(rg=rg2, side=side2) == -1, kw
    rg3, side3 = _structs(len_xform=2)
    assert call(rg=rg3, side=side3) == -3
    # the inputs a wanted gradient needs
    for kw in (dict(g=None), dict(x=None), dict(dl=None), dict(A=None), dict(Bm=None), dict(Cm=None), dict(st=None)):
        assert call(**kw) == -1, kw
    # grad_A / grad_B without (enough) workspace
    assert call(ga=ga) == -2 and call(gb=ga) == -2
    need = lib.rua_ssm_workspace_bytes(4, 2, 8, 4, 0)
    assert call(ga=ga, ws=0x9000, nbytes=need - 1) == -2
    # nothing wanted: OK
    assert call(gx=None) == 0


@pytest.mark.parametrize('dtype', range(4))
def test_ssm_state_and_workspace_bounds(lib, dtype):
    state, ws = lib.rua_ssm_state_bytes, lib.rua_ssm_workspace_bytes
    for bad in ((-1, 2, 8, 4, dtype), (8, -1, 8, 4, dtype), (8, 2, -1, 4, dtype), (8, 2, 8, 0, dtype),
                (8, 2, 8, 17, dtype), (8, 2, 8, 4, 4), (8, 2, 8, 4, -1)):
        assert state(*bad) == 0 and ws(*bad) == 0, bad
    acc = 8 if dtype == 1 else 4
    W = 64 if dtype == 1 else 128
    for B in (1, 7, 4096):
        for H in (1, 100, 1024, 4096):
            for N in (1, 3, 4, 5, 8, 9, 16):
                rows_list = [B, B + 31, B * 32, B * 512, B * 4096]
                st = [state(r, B, H, N, dtype) for r in rows_list]
                w = [ws(r, B, H, N, dtype) for r in rows_list]
                assert st == sorted(st) and w == sorted(w) and all(v > 0 for v in st + w)
                nblk = math.ceil(H / W)
                for r, s_, w_ in zip(rows_list, st, w):
                    # one H x N state per 32 tokens plus one per sequence
                    assert s_ <= (r // 32 + B) * H * N * acc
                    # grad_A slots for at most 8 CTAs per SM, and one [grad_B | grad_C] partial per (token, block)
                    slots = min(B, math.ceil(148 * 8 / nblk)) * H * N * acc
                    assert w_ <= (slots + 255) // 256 * 256 + nblk * r * 2 * N * acc
                    assert w_ >= nblk * r * 2 * N * acc
    assert ws(0, 2, 8, 4, dtype) == 0 and ws(8, 0, 8, 4, dtype) == 0 and ws(8, 2, 0, 4, dtype) == 0


def test_ssm_python_rejects_bad_arguments():
    import torchrua_b200 as rua
    lens = torch.tensor([2, 3])
    x, d = torch.randn(5, 6), torch.rand(5, 6)
    A, Bm, Cm = -torch.rand(6, 4), torch.randn(5, 4), torch.randn(5, 4)
    # CPU tensors
    for call in (lambda: rua.segment_selective_scan(x, lens, d, A, Bm, Cm),
                 lambda: rua.C(data=x, token_sizes=lens).selective_scan(d, A, Bm, Cm),
                 lambda: rua.L(data=torch.randn(2, 3, 6), token_sizes=lens).selective_scan(
                     torch.rand(2, 3, 6), A, torch.randn(2, 3, 4), torch.randn(2, 3, 4))):
        with pytest.raises(RuntimeError, match='CUDA tensors only'):
            call()
    # integer payloads, mismatched dtypes
    with pytest.raises(RuntimeError, match='float16/bfloat16/float32/float64'):
        rua.segment_selective_scan(x.long(), lens, d.long(), A, Bm, Cm)
    with pytest.raises(RuntimeError, match='delta must have dtype'):
        rua.segment_selective_scan(x, lens, d.double(), A, Bm, Cm)
    with pytest.raises(RuntimeError, match='B must have dtype'):
        rua.segment_selective_scan(x, lens, d, A, Bm.half(), Cm)
    with pytest.raises(RuntimeError, match='C must have dtype'):
        rua.segment_selective_scan(x, lens, d, A, Bm, Cm.double())
    with pytest.raises(RuntimeError, match='A must have dtype'):   # A is fp32 for a bf16 payload
        rua.segment_selective_scan(x.bfloat16(), lens, d.bfloat16(), A.bfloat16(), Bm.bfloat16(), Cm.bfloat16())
    with pytest.raises(RuntimeError, match='initial must have dtype'):
        rua.segment_selective_scan(x, lens, d, A, Bm, Cm, torch.zeros(2, 6, 4, dtype=torch.float64))
    # shapes
    with pytest.raises(ValueError, match='delta must have the shape'):
        rua.segment_selective_scan(x, lens, d[:, :5], A, Bm, Cm)
    for b in (torch.randn(4, 4), torch.randn(5), torch.randn(5, 4, 1)):
        with pytest.raises(ValueError, match='B must be'):
            rua.segment_selective_scan(x, lens, d, A, b, Cm)
    with pytest.raises(ValueError, match='C must have the shape of B'):
        rua.segment_selective_scan(x, lens, d, A, Bm, torch.randn(5, 3))
    for a in (torch.randn(6, 3), torch.randn(5, 4), torch.randn(4)):
        with pytest.raises(ValueError, match=r'A must be \(\*feat, N\)'):
            rua.segment_selective_scan(x, lens, d, a, Bm, Cm)
    for h0 in (torch.zeros(3, 6, 4), torch.zeros(2, 6), torch.zeros(2, 6, 3)):
        with pytest.raises(ValueError, match='initial must be'):
            rua.segment_selective_scan(x, lens, d, A, Bm, Cm, h0)
    # state sizes outside [1, 16]
    for N in (0, 17, 32):
        with pytest.raises(ValueError, match='state sizes 1..16'):
            rua.segment_selective_scan(x, lens, d, torch.randn(6, N), torch.randn(5, N), torch.randn(5, N))
    with pytest.raises(ValueError, match='B must be'):
        rua.L(data=torch.randn(2, 3, 6), token_sizes=lens).selective_scan(torch.rand(2, 3, 6), A, Bm, Cm)


def test_ssm_names_are_exported():
    import torchrua
    import torchrua.ssm
    import torchrua_b200 as rua
    assert torchrua.segment_selective_scan is rua.segment_selective_scan
    assert torchrua.ssm.segment_selective_scan is rua.segment_selective_scan
    for cls in (rua.C, rua.L, rua.P, rua.R):
        assert callable(cls.selective_scan)
