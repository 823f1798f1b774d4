"""CPU-only checks of the gated delta rule boundary: argument validation happens before any CUDA call, the documented
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


def test_gdn_forward_validates_before_cuda(lib):
    fwd, ref = lib.rua_gdn_forward, ctypes.byref
    rg, side = _structs()
    v, q, k, g, b, o = (0x1000 * j for j in range(1, 7))

    def call(v=v, q=q, k=k, g=g, b=b, o=o, H=8, G=2, K=4, V=4, dtype=0, reverse=0, rg=rg, side=side):
        return fwd(v, q, k, g, b, None, o, None, H, G, K, V, 0.5, dtype, reverse, None if rg is None else ref(rg),
                   None if side is None else ref(side), None, 0, None)

    assert call(rg=None) == -1 and call(side=None) == -1
    for dtype in (-1, 4, 7):
        assert call(dtype=dtype) == -1
    assert call(K=0) == -1 and call(V=0) == -1 and call(G=0) == -1 and call(K=-3) == -1
    assert call(G=3) == -1 and call(H=6, G=4) == -1   # H % G != 0
    assert call(K=129) == -3 and call(V=257) == -3 and call(K=256, V=512) == -3
    assert call(H=-1) == -1 and call(reverse=2) == -1 and call(reverse=-1) == -1
    for kw in BAD_LAYOUTS:
        rg2, side2 = _structs(**kw)
        assert call(rg=rg2, side=side2) == -1, kw
    rg3, side3 = _structs(len_xform=1)
    assert call(rg=rg3, side=side3) == -3
    for kw in (dict(v=None), dict(q=None), dict(k=None), dict(g=None), dict(b=None), dict(o=None)):
        assert call(**kw) == -1, kw
    rg4, side4 = _structs(B=0, rows=0)
    assert fwd(None, None, None, None, None, None, None, None, 8, 2, 4, 4, 0.5, 0, 0, ref(rg4), ref(side4), None, 0,
               None) == 0
    assert call(H=0) == 0


def test_gdn_backward_validates_before_cuda(lib):
    bwd, ref = lib.rua_gdn_backward, ctypes.byref
    rg, side = _structs()
    go, v, q, k, g, b, gv, gg = (0x1000 * j for j in range(1, 9))
    need = lib.rua_gdn_workspace_bytes(4, 2, 4, 8, 2, 4, 4, 0)

    def call(go=go, v=v, q=q, k=k, g=g, b=b, gv=gv, gg=None, H=8, G=2, K=4, V=4, dtype=0, reverse=0, rg=rg,
             side=side, ws=0x9000, nbytes=need):
        return bwd(go, v, q, k, g, b, None, gv, None, None, gg, None, None, H, G, K, V, 0.5, dtype, reverse,
                   None if rg is None else ref(rg), None if side is None else ref(side), ws, nbytes, None)

    assert call(rg=None) == -1 and call(side=None) == -1
    assert call(dtype=5) == -1 and call(K=0) == -1 and call(V=0) == -1 and call(reverse=3) == -1
    assert call(G=3) == -1 and call(K=129) == -3 and call(V=257) == -3
    for kw in BAD_LAYOUTS:
        rg2, side2 = _structs(**kw)
        assert call(rg=rg2, side=side2) == -1, kw
    rg3, side3 = _structs(len_xform=2)
    assert call(rg=rg3, side=side3) == -3
    for kw in (dict(go=None), dict(v=None), dict(q=None), dict(k=None), dict(g=None), dict(b=None)):
        assert call(**kw) == -1, kw
    assert need > 0
    assert call(ws=None) == -2 and call(nbytes=need - 1) == -2 and call(gg=gg, ws=None) == -2
    assert call(gv=None) == 0
    rg4, side4 = _structs(B=0, rows=0)
    assert call(rg=rg4, side=side4, ws=None, nbytes=0) == 0
    assert call(H=0, ws=None, nbytes=0) == 0


@pytest.mark.parametrize('dtype', range(4))
def test_gdn_workspace_formula_and_monotone(lib, dtype):
    ws = lib.rua_gdn_workspace_bytes
    for bad in ((-1, 2, 4, 8, 2, 4, 4, dtype), (8, -1, 4, 8, 2, 4, 4, dtype), (8, 2, -1, 8, 2, 4, 4, dtype),
                (8, 2, 4, -1, 2, 4, 4, dtype), (8, 2, 4, 8, 0, 4, 4, dtype), (8, 2, 4, 8, 3, 4, 4, dtype),
                (8, 2, 4, 8, 2, 0, 4, dtype), (8, 2, 4, 8, 2, 129, 4, dtype), (8, 2, 4, 8, 2, 4, 0, dtype),
                (8, 2, 4, 8, 2, 4, 257, dtype), (8, 2, 4, 8, 2, 4, 4, 4), (8, 2, 4, 8, 2, 4, 4, -1)):
        assert ws(*bad) == 0, bad
    assert ws(0, 2, 4, 8, 2, 4, 4, dtype) == 0 and ws(8, 0, 4, 8, 2, 4, 4, dtype) == 0
    assert ws(8, 2, 4, 0, 2, 4, 4, dtype) == 0
    acc = 8 if dtype == 1 else 4
    Q = {0: 32, 1: 16, 2: 64, 3: 64}[dtype]
    VB = 32 if dtype == 1 else 64

    def formula(rows, B, T, H, G, K, V):
        grid = min(B * G, 296)
        return grid * (math.ceil(T / Q) * K * VB + T * (2 * K + 2)) * acc

    base = dict(rows=4096, B=16, T=1000, H=16, G=2, K=64, V=64)
    steps = dict(rows=(1, 100, 4096, 10 ** 6), B=(1, 7, 16, 40, 1000), T=(0, 1, 63, 64, 65, 4096),
                 H=(2, 4, 16, 64, 256), G=(1, 2), K=(1, 7, 64, 65, 128), V=(1, 5, 64, 65, 256))
    for key, values in steps.items():
        got = []
        for val in values:
            args = dict(base, **{key: val})
            w = ws(args['rows'], args['B'], args['T'], args['H'], args['G'], args['K'], args['V'], dtype)
            assert w == formula(*args.values()), args
            got.append(w)
        assert got == sorted(got), (key, got)
    got = [ws(4096, 16, 1000, 24, G, 64, 64, dtype) for G in (1, 2, 3, 4, 6, 8, 12, 24)]
    assert got == sorted(got)
    # about 1.87 GB at cfg3 (Tmax = 4096, K = 128, 296 CTAs) for the 16-bit payloads
    if dtype in (2, 3):
        assert 1.0e9 < ws(10 ** 6, 1000, 4096, 32, 16, 128, 128, dtype) < 2.5e9


def test_gdn_python_rejects_bad_arguments():
    import torchrua_b200 as rua
    lens = torch.tensor([2, 3])
    v, q, k = torch.randn(5, 4, 3), torch.randn(5, 2, 8), torch.randn(5, 2, 8)
    g, b = -torch.rand(5, 4), torch.rand(5, 4)
    with pytest.raises(RuntimeError, match='CUDA'):
        rua.segment_gated_delta_rule(v, lens, q, k, g, b)
    with pytest.raises(RuntimeError, match='supports float16'):
        rua.segment_gated_delta_rule(v.long(), lens, q, k, g, b)
    with pytest.raises(RuntimeError, match='q must have dtype'):
        rua.segment_gated_delta_rule(v, lens, q.double(), k, g, b)
    with pytest.raises(RuntimeError, match='beta must have dtype'):
        rua.segment_gated_delta_rule(v.half(), lens, q.half(), k.half(), g, b)
    with pytest.raises(RuntimeError, match='g must have dtype'):
        rua.segment_gated_delta_rule(v.half(), lens, q.half(), k.half(), g.half(), b.half())
    with pytest.raises(RuntimeError, match='initial must have dtype'):
        rua.segment_gated_delta_rule(v, lens, q, k, g, b, initial=torch.zeros(2, 4, 8, 3, dtype=torch.float64))
    with pytest.raises(ValueError, match=r'row dimension\(s\) \+ \(H, V\)'):
        rua.segment_gated_delta_rule(v[:, 0], lens, q, k, g, b)
    with pytest.raises(ValueError, match='q must be'):
        rua.segment_gated_delta_rule(v, lens, q[:4], k, g, b)
    with pytest.raises(ValueError, match='k must have the shape of q'):
        rua.segment_gated_delta_rule(v, lens, q, k[:, :1], g, b)
    with pytest.raises(ValueError, match='g must be'):
        rua.segment_gated_delta_rule(v, lens, q, k, g[:, :3], b)
    with pytest.raises(ValueError, match='beta must be'):
        rua.segment_gated_delta_rule(v, lens, q, k, g, b[:4])
    with pytest.raises(ValueError, match='to split into G = 3'):
        rua.segment_gated_delta_rule(v, lens, torch.randn(5, 3, 8), torch.randn(5, 3, 8), g, b)
    with pytest.raises(ValueError, match='key dims 1..128'):
        rua.segment_gated_delta_rule(v, lens, torch.randn(5, 2, 129), torch.randn(5, 2, 129), g, b)
    with pytest.raises(ValueError, match='value dims 1..256'):
        rua.segment_gated_delta_rule(torch.randn(5, 4, 257), lens, q, k, g, b)
    with pytest.raises(ValueError, match='initial must be'):
        rua.segment_gated_delta_rule(v, lens, q, k, g, b, initial=torch.zeros(2, 4, 3, 8))
    with pytest.raises(ValueError, match='q must be'):
        rua.L(data=torch.randn(2, 3, 4, 3), token_sizes=lens).gated_delta_rule(q, k, g, b)


def test_gdn_scale_default():
    from torchrua_b200 import _native
    assert _native.gdn_scale(None, 128) == 128 ** -0.5 and _native.gdn_scale(0.25, 128) == 0.25


def test_gdn_names_are_exported():
    import torchrua
    import torchrua.delta
    import torchrua_b200 as rua
    assert torchrua.segment_gated_delta_rule is rua.segment_gated_delta_rule
    assert torchrua.delta.segment_gated_delta_rule is rua.segment_gated_delta_rule
    for cls in (rua.C, rua.L, rua.P, rua.R):
        assert callable(cls.gated_delta_rule)
