"""CPU-only checks of the linear-chain CRF boundary: argument validation happens before any CUDA call, the workspace
rule, and the Python entry points reject bad dtypes, shapes, tag counts, tags and CPU tensors before device work."""
import ctypes

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


def test_crf_forward_validates_before_cuda(lib):
    fwd, ref = lib.rua_crf_forward, ctypes.byref
    rg, side = _structs()
    x, tags, W, lz, sc = 0x1000, 0x2000, 0x3000, 0x4000, 0x5000

    def call(x=x, tags=None, W=W, lz=lz, sc=None, K=4, dtype=0, rg=rg, side=side):
        return fwd(x, tags, W, None, None, lz, sc, None, K, dtype, None if rg is None else ref(rg),
                   None if side is None else ref(side), None, 0, None)

    assert call(rg=None) == -1 and call(side=None) == -1
    for dtype in (-1, 4, 7):
        assert call(dtype=dtype) == -1
    assert call(K=0) == -1 and call(K=-3) == -1
    assert call(K=65) == -3 and call(K=1000) == -3
    for kw in BAD_LAYOUTS:
        rg2, side2 = _structs(**kw)
        assert call(rg=rg2, side=side2) == -1, kw
    rg3, side3 = _structs(len_xform=1)
    assert call(rg=rg3, side=side3) == -3
    # missing buffers; tags and score come together
    assert call(x=None) == -1 and call(W=None) == -1 and call(lz=None) == -1
    assert call(tags=tags) == -1 and call(sc=sc) == -1
    # nothing to do: OK without touching anything
    rg4, side4 = _structs(B=0, rows=0)
    assert fwd(None, None, None, None, None, None, None, None, 4, 0, ref(rg4), ref(side4), None, 0, None) == 0


def test_crf_backward_validates_before_cuda(lib):
    bwd, ref = lib.rua_crf_backward, ctypes.byref
    rg, side = _structs()
    gz, gs, x, tags, W, st, lz, gx, gw = (0x1000 * k for k in range(1, 10))

    def call(gz=gz, gs=None, x=x, tags=None, W=W, st=st, lz=lz, gx=gx, gw=None, K=4, dtype=0, rg=rg, side=side, ws=None,
             nbytes=0):
        return bwd(gz, gs, x, tags, W, None, None, st, lz, gx, gw, None, None, K, dtype,
                   None if rg is None else ref(rg), None if side is None else ref(side), ws, nbytes, None)

    assert call(rg=None) == -1 and call(side=None) == -1
    assert call(dtype=5) == -1 and call(K=0) == -1 and call(K=65) == -3
    for kw in BAD_LAYOUTS:
        rg2, side2 = _structs(**kw)
        assert call(rg=rg2, side=side2) == -1, kw
    # the inputs a wanted gradient needs
    for kw in (dict(gz=None), dict(x=None), dict(st=None), dict(lz=None), dict(W=None), dict(gs=gs)):
        assert call(**kw) == -1, kw
    # grad_W without (enough) workspace
    assert call(gw=gw) == -2
    need = lib.rua_crf_workspace_bytes(4, 4, 0, 1)
    assert call(gw=gw, ws=0x9000, nbytes=need - 1) == -2
    # nothing wanted: OK
    assert call(gx=None) == 0


def test_crf_decode_validates_before_cuda(lib):
    dec, ref = lib.rua_crf_decode, ctypes.byref
    rg, side = _structs()
    x, W, out, best = 0x1000, 0x2000, 0x3000, 0x4000

    def call(x=x, W=W, out=out, best=best, K=4, dtype=0, rg=rg, side=side, ws=None, nbytes=0):
        return dec(x, W, None, None, out, best, K, dtype, None if rg is None else ref(rg),
                   None if side is None else ref(side), ws, nbytes, None)

    assert call(rg=None) == -1 and call(side=None) == -1
    assert call(dtype=4) == -1 and call(K=0) == -1 and call(K=65) == -3
    for kw in BAD_LAYOUTS:
        rg2, side2 = _structs(**kw)
        assert call(rg=rg2, side=side2) == -1, kw
    for kw in (dict(x=None), dict(W=None), dict(out=None), dict(best=None)):
        assert call(**kw) == -1, kw
    assert call() == -2
    assert call(ws=0x9000, nbytes=4 * 4 - 1) == -2


def test_crf_workspace_rule(lib):
    ws, state = lib.rua_crf_workspace_bytes, lib.rua_crf_state_bytes
    for bad in ((-1, 4, 0, 1), (8, 0, 0, 1), (8, 65, 0, 1), (8, 4, 4, 1), (8, 4, -1, 2)):
        assert ws(*bad) == 0, bad
    assert ws(0, 4, 0, 1) == 0 and ws(0, 4, 0, 2) == 0
    for dtype in range(4):
        for K in (1, 2, 5, 32, 33, 64):
            assert ws(100, K, dtype, 0) == 0                      # the forward needs none
            assert ws(100, K, dtype, 2) == 100 * K                 # uint8 backpointers
            back = [ws(rows, K, dtype, 1) for rows in (1, 10, 1 << 10, 1 << 20, 1 << 30, 1 << 40)]
            assert all(b > 0 for b in back) and back == sorted(back)  # monotone ...
            assert back[-1] <= 64 << 20                            # ... and bounded
            acc = 8 if dtype == 1 else 4
            assert state(7, K, dtype) >= 7 * K * acc + 7 * 8
    assert state(0, 4, 0) == 0 and state(4, 0, 0) == 0


def test_crf_python_rejects_bad_arguments():
    import torchrua_b200 as rua
    lens = torch.tensor([2, 3])
    x, W, s = torch.randn(5, 4), torch.randn(4, 4), torch.randn(4)
    tags = torch.zeros(5, dtype=torch.long)
    # CPU tensors
    for call in (lambda: rua.segment_crf_log_partition(x, lens, W), lambda: rua.segment_crf_decode(x, lens, W, s, s),
                 lambda: rua.segment_crf_log_likelihood(x, lens, tags, W),
                 lambda: rua.C(data=x, token_sizes=lens).crf_log_partition(W),
                 lambda: rua.L(data=torch.randn(2, 3, 4), token_sizes=lens).crf_decode(W),
                 lambda: rua.R(data=torch.randn(2, 3, 4), token_sizes=lens).crf_log_likelihood(torch.zeros(2, 3).long(), W)):
        with pytest.raises(RuntimeError, match='CUDA tensors only'):
            call()
    # integer payloads, mismatched dtypes
    with pytest.raises(RuntimeError, match='float16/bfloat16/float32/float64'):
        rua.segment_crf_log_partition(torch.arange(20).view(5, 4), lens, W.long())
    with pytest.raises(RuntimeError, match='transitions has dtype'):
        rua.segment_crf_log_partition(x, lens, W.double())
    with pytest.raises(RuntimeError, match='start has dtype'):
        rua.segment_crf_log_partition(x, lens, W, s.half())
    with pytest.raises(RuntimeError, match='end has dtype'):
        rua.segment_crf_decode(x, lens, W, None, s.to(torch.bfloat16))
    # shapes
    for w in (torch.randn(4, 5), torch.randn(4), torch.randn(3, 3), torch.randn(4, 4, 1)):
        with pytest.raises(ValueError, match=r'transitions must be \(K, K\)'):
            rua.segment_crf_log_partition(x, lens, w)
    for v in (torch.randn(3), torch.randn(4, 1), torch.randn(1, 4)):
        with pytest.raises(ValueError, match=r'start must be \(K,\)'):
            rua.segment_crf_log_partition(x, lens, W, v)
        with pytest.raises(ValueError, match=r'end must be \(K,\)'):
            rua.segment_crf_log_partition(x, lens, W, None, v)
    with pytest.raises(ValueError, match='row dimension'):
        rua.segment_crf_log_partition(torch.randn(5, 4, 2), lens, W)
    with pytest.raises(ValueError, match='row dimension'):
        rua.L(data=torch.randn(2, 3), token_sizes=lens).crf_log_partition(W)
    # tag counts outside [1, 64]
    for K in (0, 65, 100):
        with pytest.raises(ValueError, match='1..64 tags'):
            rua.segment_crf_log_partition(torch.randn(5, K), lens, torch.randn(K, K))
    # tags: int64 and shaped like the rows
    for bad in (tags.int(), tags.float()):
        with pytest.raises(RuntimeError, match='tags must be int64'):
            rua.segment_crf_log_likelihood(x, lens, bad, W)
    for bad in (torch.zeros(4, dtype=torch.long), torch.zeros(5, 1, dtype=torch.long)):
        with pytest.raises(ValueError, match='tags must have the shape'):
            rua.segment_crf_log_likelihood(x, lens, bad, W)
    with pytest.raises(ValueError, match='tags must have the shape'):
        rua.L(data=torch.randn(2, 3, 4), token_sizes=lens).crf_log_likelihood(torch.zeros(6, dtype=torch.long), W)


def test_crf_names_are_exported():
    import torchrua
    import torchrua.crf
    import torchrua_b200 as rua
    for name in ('segment_crf_log_partition', 'segment_crf_log_likelihood', 'segment_crf_decode'):
        assert getattr(torchrua, name) is getattr(rua, name)
        assert getattr(torchrua.crf, name) is getattr(rua, name)
    for cls in (rua.C, rua.L, rua.P, rua.R):
        for m in ('crf_log_partition', 'crf_log_likelihood', 'crf_decode'):
            assert callable(getattr(cls, m))
