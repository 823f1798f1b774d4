"""CPU-only checks of the prefix-scan boundary: argument validation happens before any CUDA call, and the Python entry
points reject CPU tensors and integer payloads with the package's usual messages."""
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


def test_scan_entry_points_validate_before_cuda(lib):
    from torchrua_b200 import _lib
    rg, side = _structs()
    scan, bwd = lib.rua_segment_scan, lib.rua_segment_scan_backward
    ref = ctypes.byref
    # null structs, negative sizes, bad enums
    assert scan(None, None, None, 8, 0, 0, 0, None, None, None, 0, None) == -1
    assert scan(None, None, None, -1, 0, 0, 0, ref(rg), ref(side), None, 0, None) == -1
    assert scan(None, None, None, 8, 7, 0, 0, ref(rg), ref(side), None, 0, None) == -1
    assert scan(None, None, None, 8, 0, 9, 0, ref(rg), ref(side), None, 0, None) == -1
    # null buffers
    assert scan(None, None, None, 8, 0, _lib.SCAN_SUM, 0, ref(rg), ref(side), None, 0, None) == -1
    assert scan(0x1000, 0x2000, None, 8, 0, _lib.SCAN_MAX, 0, ref(rg), ref(side), None, 0, None) == -1  # no idx_out
    # negative rows, no offsets, P without its permutation, L whose rows are not B * W
    rg2, side2 = _structs(rows=-1)
    assert scan(0x1000, 0x2000, None, 8, 0, 0, 0, ref(rg2), ref(side2), None, 0, None) == -1
    rg3, side3 = _structs(off=False)
    assert scan(0x1000, 0x2000, None, 8, 0, 0, 0, ref(rg3), ref(side3), None, 0, None) == -1
    rg4, side4 = _structs(layout=_lib.PACK)
    assert scan(0x1000, 0x2000, None, 8, 0, 0, 0, ref(rg4), ref(side4), None, 0, None) == -1
    rg5, side5 = _structs(layout=_lib.LEFT, rows=5, width=3)
    assert scan(0x1000, 0x2000, None, 8, 0, 0, 0, ref(rg5), ref(side5), None, 0, None) == -1
    # a valid call with too small a workspace is refused before the memset
    assert scan(0x1000, 0x2000, None, 8, 0, 0, 0, ref(rg), ref(side), None, 0, None) == -2
    # backward: the inputs each op needs
    assert bwd(None, None, None, None, None, 8, 0, 0, 0, ref(rg), ref(side), None, 0, None) == -1
    assert bwd(0x1000, None, None, None, 0x2000, 8, 0, _lib.SCAN_LOGSUMEXP, 0, ref(rg), ref(side), None, 0, None) == -1
    assert bwd(0x1000, None, None, None, 0x2000, 8, 0, _lib.SCAN_MIN, 0, ref(rg), ref(side), None, 0, None) == -1
    assert bwd(0x1000, None, None, None, 0x2000, -3, 0, 0, 0, ref(rg), ref(side), None, 0, None) == -1
    # nothing to do: OK without touching anything
    rg6, side6 = _structs(rows=0)
    assert scan(None, None, None, 8, 0, 0, 0, ref(rg6), ref(side6), None, 0, None) == 0
    assert lib.rua_segment_scan_workspace_bytes(-1, 8, 0, 0, 0) == 0
    assert lib.rua_segment_scan_workspace_bytes(1 << 20, 1024, 3, 2, 0) > 0
    assert lib.rua_segment_scan_workspace_bytes(1 << 20, 1024, 3, 2, 1) > 0


def test_scan_python_rejects_cpu_and_integer_tensors():
    import torchrua_b200 as rua
    lens = torch.tensor([2, 3])
    for fn in (rua.segment_cumsum, rua.segment_logcumsumexp, rua.segment_cummax, rua.segment_cummin):
        with pytest.raises(RuntimeError, match='CUDA tensors only'):
            fn(torch.randn(5, 2), lens)
    c = rua.C(data=torch.randn(5, 2), token_sizes=lens)
    for call in (c.cumsum, c.logcumsumexp, c.cummax, c.cummin):
        with pytest.raises(RuntimeError, match='CUDA tensors only'):
            call()
    # integer payloads are refused before anything touches a device
    ints = rua.C(data=torch.arange(5), token_sizes=lens)
    for call in (lambda: rua.segment_cumsum(torch.arange(5), lens), lambda: rua.segment_cummax(ints.data, lens),
                 ints.cumsum, ints.logcumsumexp, ints.cummax, ints.cummin,
                 rua.L(data=torch.arange(6).view(2, 3), token_sizes=lens).cumsum,
                 rua.R(data=torch.arange(6).view(2, 3), token_sizes=lens).cummin):
        with pytest.raises(RuntimeError, match='segment scans support float'):
            call()


def test_scan_names_are_exported():
    import torchrua
    import torchrua_b200 as rua
    for name in ('segment_cumsum', 'segment_logcumsumexp', 'segment_cummax', 'segment_cummin'):
        assert getattr(torchrua, name) is getattr(rua, name)
    for cls in (rua.C, rua.L, rua.P, rua.R):
        for m in ('cumsum', 'logcumsumexp', 'cummax', 'cummin'):
            assert callable(getattr(cls, m))
