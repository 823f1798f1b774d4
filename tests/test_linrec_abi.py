"""CPU-only checks of the linear-recurrence boundary: argument validation happens before any CUDA call, the workspace
rule, and the Python entry points reject CPU tensors, integer payloads and mismatched gate / initial shapes."""
import ctypes

import pytest
import torch


@pytest.fixture(scope='module')
def lib():
    import __graft_entry__ as entry
    entry.build_cuda()
    from torchrua_b200 import _lib
    return _lib.load()


def _structs(layout=0, rows=4, width=0, B=2, off=True, pack=False, len_xform=0):
    from torchrua_b200 import _lib
    fake = 0x1000   # never dereferenced: every call below fails validation first
    rg = _lib.Ragged(B, fake if off else None, fake if pack else None, fake if pack else None,
                     fake if pack else None, 1 if pack else 0)
    return rg, _lib.Side(layout, len_xform, 0, width, rows)


def test_linrec_forward_validates_before_cuda(lib):
    from torchrua_b200 import _lib
    fwd, ref = lib.rua_segment_linrec, ctypes.byref
    rg, side = _structs()
    x, a, h0, y = 0x1000, 0x2000, 0x3000, 0x4000
    # null structs, negative H, bad dtype
    assert fwd(x, a, None, y, 8, 0, 0, None, None, None, 0, None) == -1
    assert fwd(x, a, None, y, 8, 0, 0, ref(rg), None, None, 0, None) == -1
    assert fwd(x, a, None, y, -1, 0, 0, ref(rg), ref(side), None, 0, None) == -1
    assert fwd(x, a, None, y, 8, 7, 0, ref(rg), ref(side), None, 0, None) == -1
    assert fwd(x, a, None, y, 8, -1, 0, ref(rg), ref(side), None, 0, None) == -1
    # missing buffers: x, gate, dst
    assert fwd(None, a, None, y, 8, 0, 0, ref(rg), ref(side), None, 0, None) == -1
    assert fwd(x, None, None, y, 8, 0, 0, ref(rg), ref(side), None, 0, None) == -1
    assert fwd(x, a, h0, None, 8, 0, 0, ref(rg), ref(side), None, 0, None) == -1
    # negative rows / B, no offsets, P without its permutation, L / R whose rows are not B * W, another length rule
    for kw in (dict(rows=-1), dict(B=-1), dict(off=False), dict(layout=_lib.PACK), dict(layout=_lib.LEFT, rows=5, width=3),
               dict(layout=_lib.RIGHT, rows=5, width=3), dict(layout=9)):
        rg2, side2 = _structs(**kw)
        assert fwd(x, a, None, y, 8, 0, 0, ref(rg2), ref(side2), None, 0, None) == -1, kw
    rg3, side3 = _structs(len_xform=_lib.LEN_CONST)
    assert fwd(x, a, None, y, 8, 0, 0, ref(rg3), ref(side3), None, 0, None) == -3
    # a valid call with too small a workspace is refused before the memset
    assert fwd(x, a, h0, y, 8, 0, 0, ref(rg), ref(side), None, 0, None) == -2
    # nothing to do: OK without touching anything, even with NULL buffers
    rg4, side4 = _structs(rows=0)
    assert fwd(None, None, None, None, 8, 0, 0, ref(rg4), ref(side4), None, 0, None) == 0
    assert fwd(None, None, None, None, 0, 0, 0, ref(rg), ref(side), None, 0, None) == 0


def test_linrec_backward_validates_before_cuda(lib):
    bwd, ref = lib.rua_segment_linrec_backward, ctypes.byref
    rg, side = _structs()
    g, a, h0, y, gx, gg, gh = 0x1000, 0x2000, 0x3000, 0x4000, 0x5000, 0x6000, 0x7000

    def call(*bufs, H=8, dtype=0, rg=rg, side=side):
        return bwd(*bufs, H, dtype, 0, None if rg is None else ref(rg), None if side is None else ref(side), None, 0, None)

    assert call(g, a, h0, y, gx, gg, gh, rg=None) == -1
    assert call(g, a, h0, y, gx, gg, gh, H=-2) == -1
    assert call(g, a, h0, y, gx, gg, gh, dtype=4) == -1
    # the inputs a wanted output needs: grad_out and the gate always, y for grad_gate
    assert call(None, a, h0, y, gx, None, None) == -1
    assert call(g, None, h0, y, None, None, gh) == -1
    assert call(g, a, h0, None, None, gg, None) == -1
    rgp, sidep = _structs(layout=2)
    assert call(g, a, h0, y, gx, gg, gh, rg=rgp, side=sidep) == -1
    # y is not needed without grad_gate; h0 may be NULL: then only the workspace is missing
    assert call(g, a, None, None, gx, None, gh) == -2
    # nothing wanted, or nothing to do: OK
    assert call(g, a, h0, y, None, None, None) == 0
    assert call(None, None, None, None, None, None, None) == 0
    assert call(None, None, None, None, gx, gg, gh, H=0) == 0


def test_linrec_workspace_rule(lib):
    ws = lib.rua_segment_linrec_workspace_bytes
    for bad in ((-1, 8, 0, 0), (8, -1, 0, 0), (8, 8, 4, 0), (8, 8, -1, 1)):
        assert ws(*bad) == 0, bad
    assert ws(0, 8, 0, 0) == 0 and ws(8, 0, 0, 1) == 0
    for dtype in range(4):
        for backward in (0, 1):
            for rows, H in ((1, 1), (5, 7), (1 << 20, 1024), (40000, 1)):
                assert ws(rows, H, dtype, backward) > 0
            assert ws(1 << 20, 64, dtype, backward) >= ws(1 << 10, 64, dtype, backward)


def test_linrec_python_rejects_bad_arguments():
    import torchrua_b200 as rua
    lens = torch.tensor([2, 3])
    x, gate = torch.randn(5, 4), torch.rand(5, 4)
    with pytest.raises(RuntimeError, match='CUDA tensors only'):
        rua.segment_linear_recurrence(x, lens, gate)
    with pytest.raises(RuntimeError, match='CUDA tensors only'):
        rua.segment_linear_recurrence(x, lens, gate, torch.zeros(2, 4), reverse=True)
    c = rua.C(data=x, token_sizes=lens)
    left, right = rua.L(data=torch.randn(2, 3, 4), token_sizes=lens), rua.R(data=torch.randn(2, 3, 4), token_sizes=lens)
    for z, g in ((c, gate), (left, torch.rand(2, 3, 4)), (right, torch.rand(2, 3, 4))):
        with pytest.raises(RuntimeError, match='CUDA tensors only'):
            z.linear_recurrence(g)
    # integer payloads, mismatched dtypes and shapes are refused before anything touches a device
    ints = torch.arange(5)
    for call in (lambda: rua.segment_linear_recurrence(ints, lens, ints),
                 lambda: rua.C(data=ints, token_sizes=lens).linear_recurrence(ints),
                 lambda: rua.L(data=torch.arange(6).view(2, 3), token_sizes=lens).linear_recurrence(torch.ones(2, 3))):
        with pytest.raises(RuntimeError, match='float16/bfloat16/float32/float64'):
            call()
    with pytest.raises(RuntimeError, match='gate has dtype'):
        rua.segment_linear_recurrence(x, lens, gate.double())
    with pytest.raises(RuntimeError, match='initial has dtype'):
        rua.segment_linear_recurrence(x, lens, gate, torch.zeros(2, 4, dtype=torch.float16))
    for g in (torch.rand(5, 3), torch.rand(4, 4), torch.rand(5, 4, 1)):
        with pytest.raises(ValueError, match='gate must have the shape'):
            rua.segment_linear_recurrence(x, lens, g)
    for h in (torch.zeros(3, 4), torch.zeros(4), torch.zeros(2, 4, 1)):
        with pytest.raises(ValueError, match=r'initial must be \(B, \*feat\)'):
            rua.segment_linear_recurrence(x, lens, gate, h)
    with pytest.raises(ValueError, match='gate must have the shape'):
        left.linear_recurrence(gate)
    with pytest.raises(ValueError, match='initial must be'):
        right.linear_recurrence(torch.rand(2, 3, 4), torch.zeros(5, 4))


def test_linrec_names_are_exported():
    import torchrua
    import torchrua.scan
    import torchrua_b200 as rua
    assert torchrua.segment_linear_recurrence is rua.segment_linear_recurrence
    assert torchrua.scan.segment_linear_recurrence is rua.segment_linear_recurrence
    for cls in (rua.C, rua.L, rua.P, rua.R):
        assert callable(cls.linear_recurrence)
