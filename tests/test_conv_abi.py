"""CPU-only checks of the depthwise-convolution boundary: argument validation happens before any CUDA call, the
workspace query is host-only, monotone and bounded, and the Python entry points reject bad inputs with clear errors."""
import ctypes

import pytest
import torch


@pytest.fixture(scope='module')
def lib():
    import __graft_entry__ as entry
    entry.build_cuda()
    from torchrua_b200 import _lib
    return _lib.load()


def _structs(layout=0, rows=4, width=0, B=2, off=True, pack=False):
    from torchrua_b200 import _lib
    fake = 0x1000   # never dereferenced: every call below fails validation first
    rg = _lib.Ragged(B, fake if off else None, fake if pack else None, fake if pack else None,
                     fake if pack else None, 1 if pack else 0)
    return rg, _lib.Side(layout, 0, 0, width, rows)


def test_conv_entry_points_validate_before_cuda(lib):
    from torchrua_b200 import _lib
    rg, side = _structs()
    conv, bwd = lib.rua_segment_conv, lib.rua_segment_conv_backward
    ref = ctypes.byref
    a, b, w = 0x1000, 0x2000, 0x3000

    def f(K=4, pad=3, H=8, dtype=0, rg_=rg, side_=side, src=a, weight=w, dst=b):
        return conv(src, weight, None, dst, H, dtype, K, pad, ref(rg_) if rg_ is not None else None,
                    ref(side_) if side_ is not None else None, None, 0, None)
    # K, pad, H, dtype
    assert f(K=0, pad=0) == -1
    assert f(K=33, pad=0) == -3
    assert f(K=4, pad=4) == -1
    assert f(K=4, pad=-1) == -1
    assert f(H=0) == -1
    assert f(H=-5) == -1
    assert f(dtype=4) == -1
    assert f(dtype=-1) == -1
    # null structs, side validation
    assert f(rg_=None) == -1
    assert f(side_=None) == -1
    rg2, side2 = _structs(rows=-1)
    assert f(rg_=rg2, side_=side2) == -1
    rg3, side3 = _structs(off=False)
    assert f(rg_=rg3, side_=side3) == -1
    rg4, side4 = _structs(layout=_lib.PACK)
    assert f(rg_=rg4, side_=side4) == -1
    rg5, side5 = _structs(layout=_lib.LEFT, rows=5, width=3)
    assert f(rg_=rg5, side_=side5) == -1
    rg6, side6 = _structs(layout=7)
    assert f(rg_=rg6, side_=side6) == -1
    side7 = _lib.Side(0, 1, 0, 0, 4)   # a length transform other than RUA_LEN_SAME
    assert f(side_=side7) == -3
    # null buffers when there are rows
    assert f(src=None) == -1
    assert f(weight=None) == -1
    assert f(dst=None) == -1
    # nothing to do: OK without touching anything
    rg8, side8 = _structs(rows=0)
    assert f(src=None, weight=None, dst=None, rg_=rg8, side_=side8) == 0
    # backward: grad_out and weight always, x with grad_weight; a too small workspace is refused before any launch
    args = (8, 0, 4, 3, ref(rg), ref(side))
    assert bwd(None, a, w, b, None, None, *args, None, 0, None) == -1
    assert bwd(a, a, None, b, None, None, *args, None, 0, None) == -1
    assert bwd(a, None, w, None, b, None, *args, None, 0, None) == -1
    assert bwd(a, a, w, None, b, None, *args, None, 0, None) == -2
    assert bwd(a, None, w, None, None, b, *args, None, 0, None) == -2
    assert bwd(a, a, w, b, None, None, 8, 0, 4, 4, ref(rg), ref(side), None, 0, None) == -1
    assert bwd(a, a, w, b, None, None, 8, 0, 40, 3, ref(rg), ref(side), None, 0, None) == -3
    assert bwd(a, a, w, None, None, None, *args, None, 0, None) == 0   # no gradient wanted
    assert lib.rua_launch_count() == 0


def test_conv_workspace_is_host_only_monotone_and_bounded(lib):
    q = lib.rua_segment_conv_workspace_bytes
    assert q(-1, 8, 4, 0, 1) == 0 and q(0, 8, 4, 0, 1) == 0
    assert q(100, 0, 4, 0, 1) == 0 and q(100, 8, 0, 0, 1) == 0 and q(100, 8, 33, 0, 1) == 0 and q(100, 8, 4, 9, 1) == 0
    assert q(1 << 20, 1024, 4, 3, 0) == 0   # the forward needs none
    for H, K, dt in ((1, 4, 0), (3, 31, 1), (1024, 4, 3), (1024, 31, 3), (4096, 32, 0), (64, 1, 2)):
        sizes = [q(rows, H, K, dt, 1) for rows in (1, 7, 100, 4096, 1 << 16, 1 << 20, 1 << 26, 1 << 34)]
        assert all(s > 0 for s in sizes)
        assert all(a <= b for a, b in zip(sizes, sizes[1:])), (H, K, dt, sizes)
        assert sizes[-1] == sizes[-2], (H, K, dt, sizes)   # capped: independent of rows past a point
        assert sizes[-1] <= 64 << 20, (H, K, dt, sizes)
    assert lib.rua_launch_count() == 0


def test_conv_python_rejections():
    import torchrua_b200 as rua
    lens = torch.tensor([2, 3])
    x, w = torch.randn(5, 4), torch.randn(4, 3)
    with pytest.raises(RuntimeError, match='CUDA tensors only'):
        rua.segment_depthwise_conv1d(x, lens, w, padding='causal')
    for z in (rua.C(data=x, token_sizes=lens), rua.C(data=x, token_sizes=lens).to(dtype=torch.float)):
        with pytest.raises(RuntimeError, match='CUDA tensors only'):
            z.depthwise_conv1d(w, padding='same')
    with pytest.raises(RuntimeError, match='CUDA tensors only'):
        rua.L(data=torch.randn(2, 3, 4), token_sizes=lens).depthwise_conv1d(w, padding=0)
    # integer payloads, dtype mismatches, shapes, kernel sizes and padding are refused before anything touches a device
    calls = {
        'supports float': [lambda: rua.segment_depthwise_conv1d(torch.arange(5).view(5, 1), lens,
                                                               torch.ones(1, 3, dtype=torch.long), padding='causal')],
        'weight has dtype': [lambda: rua.segment_depthwise_conv1d(x, lens, w.double(), padding='causal')],
        'bias has dtype': [lambda: rua.segment_depthwise_conv1d(x, lens, w, torch.zeros(4, dtype=torch.half),
                                                                padding='causal')],
        'weight must be': [lambda: rua.segment_depthwise_conv1d(x, lens, torch.randn(3, 3), padding='causal'),
                           lambda: rua.segment_depthwise_conv1d(x, lens, torch.randn(4), padding='causal'),
                           lambda: rua.segment_depthwise_conv1d(x, lens, torch.randn(4, 1, 3), padding='causal')],
        'bias must be': [lambda: rua.segment_depthwise_conv1d(x, lens, w, torch.zeros(3), padding='causal')],
        'kernel sizes': [lambda: rua.segment_depthwise_conv1d(x, lens, torch.randn(4, 33), padding='causal'),
                         lambda: rua.segment_depthwise_conv1d(x, lens, torch.randn(4, 0), padding='causal')],
        'padding must be': [lambda: rua.segment_depthwise_conv1d(x, lens, w, padding='valid'),
                            lambda: rua.segment_depthwise_conv1d(x, lens, w, padding=3),
                            lambda: rua.segment_depthwise_conv1d(x, lens, w, padding=-1),
                            lambda: rua.segment_depthwise_conv1d(x, lens, w, padding=1.0),
                            lambda: rua.segment_depthwise_conv1d(x, lens, w, padding=True)],
    }
    for msg, fns in calls.items():
        for fn in fns:
            with pytest.raises((RuntimeError, ValueError), match=msg):
                fn()
    with pytest.raises(TypeError):
        rua.segment_depthwise_conv1d(x, lens, w)   # no default padding


def test_conv_names_are_exported():
    import torchrua
    import torchrua_b200 as rua
    assert torchrua.segment_depthwise_conv1d is rua.segment_depthwise_conv1d
    import torchrua.conv  # noqa: F401
    for cls in (rua.C, rua.L, rua.P, rua.R):
        assert callable(cls.depthwise_conv1d)
