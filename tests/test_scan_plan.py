"""CPU check of tests/scan_plan.py, the Python copy of the prefix-scan launch plan: its workspace size equals what
rua_segment_scan_workspace_bytes / rua_segment_linrec_workspace_bytes report over a grid of rows, H, dtype, operator and
direction, so the regimes test_gpu_scan_backward.py names are the ones the kernel runs."""
import itertools

import pytest
import torch

from tests import scan_plan

ROWS = [1, 7, 128, 129, 4096, 70001, 1 << 20]
HS = [1, 2, 3, 7, 8, 16, 64, 127, 128, 300, 1024, 1025, 4096]


@pytest.fixture(scope='module')
def lib():
    import __graft_entry__ as entry
    entry.build_cuda()
    from torchrua_b200 import _lib
    return _lib.load()


def test_workspace_matches_the_library(lib):
    from torchrua_b200 import _lib
    codes = {torch.float32: _lib.F32, torch.float64: _lib.F64, torch.float16: _lib.F16, torch.bfloat16: _lib.BF16}
    ops = {'sum': _lib.SCAN_SUM, 'logsumexp': _lib.SCAN_LOGSUMEXP, 'max': _lib.SCAN_MAX, 'min': _lib.SCAN_MIN}
    n = 0
    for dtype, rows, H in itertools.product(scan_plan.DTYPE, ROWS, HS):
        dt = codes[dtype]
        for op, kinds in scan_plan.SCAN_KINDS.items():
            for backward, kind in enumerate(kinds):
                got = lib.rua_segment_scan_workspace_bytes(rows, H, dt, ops[op], backward)
                assert got == scan_plan.workspace_bytes(kind, rows, H, dtype), (op, backward, dtype, rows, H)
                n += 1
        for backward, kind in enumerate(('linrec', 'linrec_bwd')):
            got = lib.rua_segment_linrec_workspace_bytes(rows, H, dt, backward)
            assert got == scan_plan.workspace_bytes(kind, rows, H, dtype), ('linrec', backward, dtype, rows, H)
            n += 1
    assert n == 3640


def test_regimes():
    """the widths the GPU cases use land where their names say"""
    P = scan_plan.plan
    for dtype in scan_plan.DTYPE:
        VV = scan_plan.vec_width(dtype)
        assert P('sum', 1, 1, dtype)[:5] == (1, 1, 256, 4096, 1)
        assert P('linrec_bwd', 1, VV, dtype)[:5] == (VV, 1, 256, 2048, 1)
        assert P('lse_bwd', 1, 8 * VV, dtype)[:5] == (VV, 8, 32, 128, 1)
        assert P('ext', 1, 7, dtype)[:5] == (1, 8, 32, 256, 1)
        assert P('linrec', 1, 75 * VV, dtype)[:5] == (VV, 32, 8, 48, 3)
        assert P('run_bwd', 1, 301, dtype)[:5] == (1, 32, 8, 64, 10)
        assert P('sum', 1, 75 * VV, dtype, aligned=False).V == 1
    # the narrow linear-recurrence backward needs the shared-memory opt-in above 48 KB
    assert P('linrec_bwd', 1, 1, torch.float32).smem > 48 * 1024
    assert P('linrec_bwd', 1, 1, torch.float64).smem > 48 * 1024
