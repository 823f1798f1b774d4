"""Tensor-level wrappers over the C-ABI: validate -> allocate outputs with torch -> call ``rua_*`` with raw
pointers on the current CUDA stream -> wrap the result.  torch is plumbing here (device memory,
streams, autograd graph); every byte of the hot path is moved or reduced by librua_b200.so.

No CPU path exists: non-CUDA tensors raise ``RuntimeError``.
"""
import ctypes
import itertools
import weakref
from dataclasses import dataclass, field
from typing import Optional, Tuple

import numpy as np
import torch
from torch import Tensor

from torchrua_b200 import _lib
from torchrua_b200._lib import (CAT, LEFT, LEN_CONST, LEN_MINUS, LEN_SAME, MAP_REV, MAP_ROLL, MAP_SHIFT, PACK,
                                PAD_FILL, PAD_ROW0, PAD_WRAP, RIGHT)

_DTYPES = {torch.float32: _lib.F32, torch.float64: _lib.F64, torch.float16: _lib.F16, torch.bfloat16: _lib.BF16}
_OPS = {'sum': _lib.SUM, 'mean': _lib.MEAN, 'prod': _lib.PROD, 'max': _lib.MAX, 'min': _lib.MIN,
        'logsumexp': _lib.LOGSUMEXP}


def require_cuda(*tensors: Tensor) -> torch.device:
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError(
                'torchrua_b200 runs on CUDA tensors only (hand-written sm_100a kernels, no CPU fallback); '
                f'got a tensor on {t.device}')
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError(f'torchrua_b200: tensors on different devices ({dev} vs {t.device})')
    return dev


# torch.cuda.current_stream() builds a Stream object through three layers of Python (~5 us; it used to be a third of the
# host time of a small call, benchmarks/diag_profile.py); the raw handle is one C call.  Private but long-lived entry points
# (inductor and triton use them); the public route stays as the fallback.
_RAW_STREAM = getattr(torch._C, '_cuda_getCurrentRawStream', None)
_CUR_DEVICE = getattr(torch._C, '_cuda_getDevice', None)
if _RAW_STREAM is None or _CUR_DEVICE is None:
    _RAW_STREAM = None
    _CUR_DEVICE = torch.cuda.current_device


def _stream() -> int:
    """raw handle of the current stream of the current device"""
    if _RAW_STREAM is not None:
        return _RAW_STREAM(_CUR_DEVICE())
    return torch.cuda.current_stream().cuda_stream


FUSED_CAP = 4096   # speculative number of batch_sizes entries fetched together with (N, T)


class _NoGuard:
    def __enter__(self):
        return None

    def __exit__(self, *exc):
        return False


_NO_GUARD = _NoGuard()


def _on(device: torch.device):
    """device guard that costs nothing in the common one-process-per-GPU case (torch.cuda.device() is
    ~10 us of Python per use; these kernels run for 5 us)."""
    idx = device.index
    if idx is None or idx == _CUR_DEVICE():
        return _NO_GUARD
    return torch.cuda.device(device)


def fetch(dev_tensor: Tensor) -> Tensor:
    """small device -> host read through pinned memory, ordered on the current stream (no device-wide
    sync, no pageable staging copy)."""
    host = torch.empty(dev_tensor.shape, dtype=dev_tensor.dtype, pin_memory=True)
    with _on(dev_tensor.device):
        host.copy_(dev_tensor, non_blocking=True)
        torch.cuda.current_stream().synchronize()
    return host


def fetch_async(dev_tensor: Tensor):
    """enqueue the device -> host read and return (pinned host tensor, event); ``event.synchronize()`` waits for
    the copy only, not for kernels enqueued after it."""
    host = torch.empty(dev_tensor.shape, dtype=dev_tensor.dtype, pin_memory=True)
    with _on(dev_tensor.device):
        host.copy_(dev_tensor, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
    return host, ev


def upload(host_tensor: Tensor, device: torch.device) -> Tensor:
    """small host -> device write through pinned memory (asynchronous, stream-ordered)."""
    pinned = torch.empty(host_tensor.shape, dtype=host_tensor.dtype, pin_memory=True)
    pinned.copy_(host_tensor)
    return pinned.to(device, non_blocking=True)


# optional per-launch timing (bench.py sets PROFILE = [] to collect (name, start, end, algorithmic_bytes);
# events are recorded on the launching stream right around the kernel launch)
PROFILE = None


def _profile_begin():
    if PROFILE is None:
        return None
    ev = torch.cuda.Event(enable_timing=True)
    ev.record()
    return ev


def _profile_end(start, name: str, nbytes: int) -> None:
    end = torch.cuda.Event(enable_timing=True)
    end.record()
    PROFILE.append((name, start, end, nbytes))


def _ptr(t: Optional[Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _i64(t: Tensor) -> Tensor:
    t = t.detach()
    if t.dtype != torch.long:
        t = t.long()
    return t.contiguous()


_SCALAR_BYTES = {}


def scalar_bytes(value, dtype: torch.dtype) -> bytes:
    """the in-memory image of ``value`` cast to ``dtype`` (fill / zero / one patterns); memoised, since
    building a one-element tensor costs more host time than launching the kernel that uses it."""
    key = (type(value), value, dtype)
    try:
        return _SCALAR_BYTES[key]
    except (KeyError, TypeError):
        pass
    if isinstance(value, Tensor):
        value = value.item()
        key = (type(value), value, dtype)
    out = bytes(torch.tensor([value], dtype=dtype).view(torch.uint8).tolist())
    if len(_SCALAR_BYTES) < 1024:
        _SCALAR_BYTES[key] = out
    return out


# ------------------------------------------------------------------------------------------------
# K0: metadata
# ------------------------------------------------------------------------------------------------
INT64_MAX = (1 << 63) - 1


class _Notices:
    """ring of [sum, max, ticket] slots in pinned host memory that the scan kernel writes directly (UVA mapping): the
    host learns N and T by polling a cache line -- no device->host copy to enqueue, no stream synchronisation.  A slot is
    reused after RING scans; a reader that finds a newer ticket falls back to copying the device-side stats."""
    RING = 512
    SPINS = 400000          # ~50 ms of polling before falling back to a stream synchronisation

    def __init__(self):
        lib = _lib.load()
        host, dev = ctypes.c_void_p(), ctypes.c_void_p()
        _lib.check(lib.rua_pinned_alloc(24 * self.RING, ctypes.byref(host), ctypes.byref(dev)), 'rua_pinned_alloc')
        self.host, self.dev = host.value, dev.value
        self.slots = [(ctypes.c_int64 * 3).from_address(self.host + 24 * k) for k in range(self.RING)]
        self.issued = 0
        self._tickets = itertools.count(1)      # next() on it is atomic under the GIL: two threads never share a ticket

    def take(self):
        ticket = next(self._tickets)
        self.issued = ticket
        k = (ticket - 1) % self.RING
        return self.slots[k], self.dev + 24 * k, ticket         # (host view, device address, ticket)

    @classmethod
    def read(cls, note):
        """-> (sum, max) or None (slot reused / timed out: use the device-side stats)."""
        slot, ticket = note
        ring = _NOTICES
        if ring is None or ring.issued - ticket >= cls.RING - 16:
            return None                 # the slot has been (or is about to be) handed to a newer scan: its words may change under us
        for _ in range(cls.SPINS):
            seen = slot[2]
            if seen == ticket:
                return slot[0], slot[1]
            if seen > ticket:
                return None
        return None


_NOTICES = None


def scan(sizes: Optional[Tensor], clamp_max: int = INT64_MAX, notify: bool = False, pack=None):
    """(off[n+1], stats[2] = (sum, max)) of an int64 device vector; no host sync.

    ``notify``: also returns a notice (third result) through which the host can read (sum, max) as soon as the kernel
    has written them to pinned host memory.  ``pack = (bs_dev, unsorted, Tp, n)``: the vector is not given but derived
    on the fly as the lengths of a PackedSequence (fourth result: the lengths) -- one launch instead of two."""
    global _NOTICES
    lib = _lib.load()
    if pack is None:
        sizes = _i64(sizes)
        require_cuda(sizes)
        n, dev = sizes.numel(), sizes.device
    else:
        bs_dev, unsorted, tp, n = pack
        dev = unsorted.device
    tiles = (n + 1023) // 1024 + 1          # >= rua_scan_workspace_bytes(n) / 8 (1024 lengths per CTA above 4096)
    note = None
    with _on(dev):
        # one allocation: [off (n+1) | stats (2) | tile status words + completion counter (tiles) | lengths (n, pack only)]
        extra = n if pack is not None else 0
        buf = torch.empty(n + 3 + tiles + extra, dtype=torch.long, device=dev)
        base = buf.data_ptr()
        note_dev, ticket = None, 0
        if notify:
            if _NOTICES is None:
                _NOTICES = _Notices()
            slot, note_dev, ticket = _NOTICES.take()
            note = (slot, ticket)
        if pack is None:
            _lib.check(lib.rua_scan_lengths_ex(sizes.data_ptr(), n, clamp_max, base, base + 8 * (n + 1), base + 8 * (n + 3),
                                               8 * tiles, None, None, 0, None, note_dev, ticket, _stream()),
                       'rua_scan_lengths_ex')
        else:
            _lib.check(lib.rua_scan_lengths_ex(None, n, clamp_max, base, base + 8 * (n + 1), base + 8 * (n + 3), 8 * tiles,
                                               bs_dev.data_ptr() if tp else None, unsorted.data_ptr(), tp,
                                               base + 8 * (n + 3 + tiles), note_dev, ticket, _stream()),
                       'rua_scan_lengths_ex')
    # (narrow, not slicing: Tensor.__getitem__ is patched process-wide -- as in the reference -- and costs ~2 us per use)
    off, stats = buf.narrow(0, 0, n + 1), buf.narrow(0, n + 1, 2)
    if pack is not None:
        return off, stats, note, buf.narrow(0, n + 3 + tiles, n)
    if notify:
        return off, stats, note
    return off, stats


def scan_with_totals(sizes: Tensor) -> Tuple[Tensor, int, int]:
    """(off[n+1], sum, max) with the two totals on the HOST (read from the scan's pinned-memory notice)."""
    off, stats, note = scan(sizes, notify=True)
    got = _Notices.read(note)
    if got is None:
        got = fetch(stats).tolist()
    return off, int(got[0]), int(got[1])


@dataclass
class Ragged:
    """device-side description of a ragged batch (base lengths) shared by every kernel call."""
    device: torch.device
    B: int
    len: Tensor                      # (B,) int64
    off: Tensor                      # (B+1,) int64
    stats: Optional[Tensor] = None   # (2,) int64 on device: (N, T)
    _N: Optional[int] = None
    _T: Optional[int] = None
    # pack side
    sorted: Optional[Tensor] = None
    unsorted: Optional[Tensor] = None
    bs_dev: Optional[Tensor] = None   # (Tp,)
    poff: Optional[Tensor] = None     # (Tp+1,)
    bs_cpu: Optional[Tensor] = None
    Tp: int = 0
    _keep: list = field(default_factory=list)
    _spec_ok: bool = False            # the speculative early launch of _ensure_pack_fused held
    _stream: Optional[int] = None     # the stream the producer kernels were enqueued on (see _cache_get)
    _note: Optional[tuple] = None     # (pinned host slot, ticket) of the scan's completion notice

    def mark_ready(self):
        with _on(self.device):
            self._stream = _stream()

    def _sync_stats(self):
        # the one inherent device -> host dependency: output shapes depend on device data.  The scan kernel has written
        # (N, T) into pinned host memory on its own; poll that, and only copy the stats back if the notice is gone.
        got = _Notices.read(self._note) if self._note is not None else None
        if got is None:
            got = fetch(self.stats).tolist()
        self._N, self._T = int(got[0]), int(got[1])

    @property
    def N(self) -> int:
        if self._N is None:
            self._sync_stats()
        return self._N

    @property
    def T(self) -> int:
        if self._T is None:
            self._sync_stats()
        return self._T

    def c_struct(self) -> _lib.Ragged:
        return _lib.Ragged(self.B, _ptr(self.off), _ptr(self.poff), _ptr(self.sorted), _ptr(self.unsorted), self.Tp)

    def ensure_pack(self) -> 'Ragged':
        """add (sorted, unsorted, batch_sizes, poff) for a lengths-based batch: device radix sort (stable
        descending) + one binary search per time step; batch_sizes goes to the host because
        PackedSequence requires it there (torchrua/core/view.py:55)."""
        if self.sorted is not None and self.poff is not None:
            return self
        lib = _lib.load()
        dev = self.device
        if self.sorted is None and 0 < self.B <= lib.rua_meta_fused_max_batch():
            return self._ensure_pack_fused()
        T = self.T
        with _on(dev):
            if self.sorted is None:
                self.sorted = torch.empty(self.B, dtype=torch.long, device=dev)
                self.unsorted = torch.empty(self.B, dtype=torch.long, device=dev)
                nbytes = lib.rua_sort_workspace_bytes(self.B)
                ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
                _lib.check(lib.rua_sort_lengths(self.len.data_ptr(), self.B, T, self.sorted.data_ptr(),
                                                self.unsorted.data_ptr(), ws.data_ptr(), nbytes, _stream()),
                           'rua_sort_lengths')
            self.bs_dev = torch.empty(T, dtype=torch.long, device=dev)
            _lib.check(lib.rua_batch_sizes(self.len.data_ptr(), self.sorted.data_ptr(), self.B, T,
                                           self.bs_dev.data_ptr(), _stream()), 'rua_batch_sizes')
        self.poff, _ = scan(self.bs_dev)
        self.Tp = T
        self.bs_cpu = fetch(self.bs_dev).clone()
        _cache_put(self.unsorted, 'pack', self)
        return self

    def _ensure_pack_fused(self, early=None) -> 'Ragged':
        """B <= 8192: ONE kernel (scan + radix sort + batch_sizes + their prefix sums) and ONE device->host copy of
        [N, T, batch_sizes].

        ``early(self)`` (optional) is called after the kernel and the copy are ENQUEUED but before the host waits for
        them, with the pack side in a speculative state (Tp = cap time steps, poff padded with N): a consumer that
        does not need N, T or batch_sizes on the host -- the C -> P row map, whose row count is the data's --
        launches there, and the host round trip overlaps it instead of idling the GPU.  ``self._spec_ok`` tells the
        caller whether the speculation held (T <= cap)."""
        lib = _lib.load()
        dev = self.device
        cap = self._T if self._T is not None else FUSED_CAP
        self._spec_ok = False
        while True:
            with _on(dev):
                self.sorted = torch.empty(self.B, dtype=torch.long, device=dev)
                self.unsorted = torch.empty(self.B, dtype=torch.long, device=dev)
                hostbuf = torch.empty(2 + cap, dtype=torch.long, device=dev)
                poff = torch.empty(cap + 1, dtype=torch.long, device=dev)
                _lib.check(lib.rua_meta_fused(self.len.data_ptr(), self.B, self.off.data_ptr(), self.sorted.data_ptr(),
                                              self.unsorted.data_ptr(), hostbuf.data_ptr(), poff.data_ptr(), cap,
                                              _stream()), 'rua_meta_fused')
            host, ev = fetch_async(hostbuf)
            speculated = False
            if early is not None:
                self.poff, self.Tp = poff, cap
                early(self)
                early, speculated = None, True      # at most once
            ev.synchronize()
            n, t = host.narrow(0, 0, 2).tolist()
            if t <= cap:
                self._spec_ok = speculated
                break
            cap = t   # a sequence longer than the speculative cap: one more round trip, exact this time
        self._N, self._T, self.Tp = n, t, t
        self.bs_cpu = host.narrow(0, 2, t).clone()
        self.bs_dev = hostbuf.narrow(0, 2, t)
        self.poff = poff.narrow(0, 0, t + 1)
        self._keep += [hostbuf, poff]
        _cache_put(self.unsorted, 'pack', self)
        return self


_CACHE = {}
_CACHE_LIMIT = 64


def _cache_get(key_tensor: Tensor, tag: str):
    """Entries are keyed on the tensor OBJECT and its version counter: in-place writes through torch (and through this
    package's own scatter, which bumps the counter) invalidate them; writes through a raw pointer that bypass the
    counter (another framework, a C extension) do not -- call ``clear_metadata_cache()`` after those.

    The cached device arrays were produced on the stream that was current when the entry was built; a consumer on
    ANOTHER stream first waits for that stream (everything enqueued there so far: a superset of the producer
    kernels -- recording an event per entry would tax the common single-stream case by ~10 us per call)."""
    ent = _CACHE.get((id(key_tensor), tag))
    if ent is None:
        return None
    ref, version, value = ent
    if ref() is key_tensor and key_tensor._version == version:
        made_on = getattr(value, '_stream', None)
        if made_on is not None:
            if _RAW_STREAM is not None and value.device.index is not None:
                same = _RAW_STREAM(value.device.index) == made_on
            else:
                same = torch.cuda.current_stream(value.device).cuda_stream == made_on
            if not same:
                cur = torch.cuda.current_stream(value.device)
                cur.wait_stream(torch.cuda.ExternalStream(made_on, device=value.device) if made_on else
                                torch.cuda.default_stream(value.device))
        return value
    del _CACHE[(id(key_tensor), tag)]
    return None


def _cache_put(key_tensor: Tensor, tag: str, value):
    if len(_CACHE) >= _CACHE_LIMIT:
        _CACHE.pop(next(iter(_CACHE)))
    if isinstance(value, Ragged):
        value.mark_ready()
    _CACHE[(id(key_tensor), tag)] = (weakref.ref(key_tensor), key_tensor._version, value)


def clear_metadata_cache() -> None:
    _CACHE.clear()


FUSED_MAX_B = 8192   # == rua_meta_fused_max_batch()


def ragged_from_lengths(token_sizes: Tensor, want_pack: bool = False, early=None) -> Ragged:
    """lengths -> Ragged, cached per lengths tensor object + version.  One scan kernel; or, when the
    pack side is wanted and the batch is small enough, one fused kernel that produces everything."""
    hit = _cache_get(token_sizes, 'len')
    if hit is not None:
        return hit.ensure_pack() if want_pack else hit
    dev = require_cuda(token_sizes)
    lens = _i64(token_sizes)
    b = lens.numel()
    if want_pack and 0 < b <= FUSED_MAX_B:
        rg = Ragged(device=dev, B=b, len=lens, off=torch.empty(b + 1, dtype=torch.long, device=dev))
        rg._ensure_pack_fused(early)
    else:
        off, stats, note = scan(lens, notify=True)
        rg = Ragged(device=dev, B=b, len=lens, off=off, stats=stats, _note=note)
        if want_pack:
            rg.ensure_pack()
    _cache_put(token_sizes, 'len', rg)
    if lens is not token_sizes:
        _cache_put(lens, 'len', rg)   # rg.len is what P -> C/L/R conversions hand out as token_sizes
    return rg


def ragged_from_pack(batch_sizes: Tensor, sorted_indices: Optional[Tensor], unsorted_indices: Optional[Tensor],
                     device: torch.device, n_rows: int) -> Ragged:
    """PackedSequence metadata -> Ragged.  No device->host sync: B, T and N are known on the host
    (batch_sizes lives there by PyTorch's contract)."""
    key = unsorted_indices if unsorted_indices is not None else batch_sizes
    hit = _cache_get(key, 'pack')
    if hit is not None and hit.bs_cpu is batch_sizes:
        return hit
    bs_cpu = batch_sizes.detach()
    if bs_cpu.is_cuda:
        bs_cpu = bs_cpu.cpu()
    if bs_cpu.dtype != torch.long or not bs_cpu.is_contiguous():
        bs_cpu = bs_cpu.long().contiguous()
    Tp = bs_cpu.numel()
    # [batch_sizes | poff] assembled with numpy straight in pinned memory (a handful of ~1 us calls instead of ~4 us
    # torch ops), then ONE asynchronous H2D
    pinned = torch.empty(2 * Tp + 1, dtype=torch.long, pin_memory=True)
    host = pinned.numpy()
    if Tp:
        bs_np = bs_cpu.numpy()
        host[:Tp] = bs_np
        host[Tp] = 0
        np.cumsum(bs_np, out=host[Tp + 1:])
        total = int(host[-1])
    else:
        host[0] = 0
        total = 0
    if n_rows >= 0 and total != n_rows:   # host-only check: inconsistent metadata would index past the payload
        raise RuntimeError(f'torchrua_b200: PackedSequence has {n_rows} rows of data but batch_sizes sums to {total}')
    # B counts every sequence, including empty ones that never show up in batch_sizes
    B = unsorted_indices.numel() if unsorted_indices is not None else (int(host[0]) if Tp > 0 else 0)
    with _on(device):
        devbuf = pinned.to(device, non_blocking=True)
        bs_dev, poff = devbuf.narrow(0, 0, Tp), devbuf.narrow(0, Tp, Tp + 1)
        if unsorted_indices is None:   # enforce_sorted=True packs carry no permutation: identity
            unsorted = torch.arange(B, dtype=torch.long, device=device)
            srt = unsorted
        else:
            unsorted = _i64(unsorted_indices)
            srt = _i64(sorted_indices)
        require_cuda(unsorted, srt)
    # lengths of the P (one binary search per sequence) and their prefix sum in ONE launch
    off, stats, _, lens = scan(None, pack=(bs_dev, unsorted, Tp, B))
    rg = Ragged(device=device, B=B, len=lens, off=off, stats=stats, _N=total, _T=Tp,
                sorted=srt, unsorted=unsorted, bs_dev=bs_dev, poff=poff, bs_cpu=batch_sizes, Tp=Tp)
    rg._keep.append(devbuf)
    _cache_put(key, 'pack', rg)
    _cache_put(lens, 'len', rg)   # token_sizes handed out by P -> C/L/R conversions resolve to this entry
    return rg


def with_injected_pack(rg: Ragged, sorted_indices: Tensor) -> Ragged:
    """a copy of ``rg`` whose pack side uses an externally supplied permutation (parity mode: feed the
    reference's non-stable sorted_indices and get bit-identical P data, SURVEY.md 8c hazard 1)."""
    lib = _lib.load()
    srt = _i64(sorted_indices)
    require_cuda(srt)
    new = Ragged(device=rg.device, B=rg.B, len=rg.len, off=rg.off, stats=rg.stats, _N=rg._N, _T=rg._T)
    new.sorted = srt
    new.unsorted = torch.empty_like(srt)
    with _on(rg.device):
        _lib.check(lib.rua_invert_permutation(srt.data_ptr(), rg.B, new.unsorted.data_ptr(), _stream()),
                   'rua_invert_permutation')
    return new.ensure_pack()


def invert_permutation(perm: Tensor) -> Tensor:
    lib = _lib.load()
    require_cuda(perm)
    p = _i64(perm)
    out = torch.empty_like(p)
    with _on(p.device):
        _lib.check(lib.rua_invert_permutation(p.data_ptr(), p.numel(), out.data_ptr(), _stream()),
                   'rua_invert_permutation')
    return out


# ------------------------------------------------------------------------------------------------
# K1/K2: ragged row map (+ autograd)
# ------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class SideSpec:
    layout: int
    xform: int = LEN_SAME
    arg: int = 0
    width: int = 0
    rows: int = 0

    def c_struct(self) -> _lib.Side:
        return _lib.Side(self.layout, self.xform, self.arg, self.width, self.rows)


@dataclass(frozen=True)
class MapSpec:
    rg: Ragged
    src: SideSpec
    dst: SideSpec
    tmap: int = MAP_SHIFT
    tmap_arg: int = 0
    pad_mode: int = PAD_FILL

    def inverse(self) -> 'MapSpec':
        """the map that routes gradients back: sides swapped, token map inverted, zero padding."""
        arg = -self.tmap_arg if self.tmap in (MAP_SHIFT, MAP_ROLL) else 0
        return MapSpec(self.rg, self.dst, self.src, self.tmap, arg, PAD_FILL)


def _row_map_raw(src: Tensor, spec: MapSpec, fill: bytes, feat: Tuple[int, ...], dtype, device) -> Tensor:
    lib = _lib.load()
    rows = spec.dst.rows
    out = torch.empty((rows,) + tuple(feat), dtype=dtype, device=device)
    if rows == 0 or out.numel() == 0:
        return out
    row_bytes = out.element_size()
    for f in feat:
        row_bytes *= f
    rg = spec.rg.c_struct()
    s, d = spec.src.c_struct(), spec.dst.c_struct()
    with _on(device):
        prof = _profile_begin()
        _lib.check(lib.rua_row_map(_ptr(src), out.data_ptr(), row_bytes, ctypes.byref(rg), ctypes.byref(s),
                                   ctypes.byref(d), spec.tmap, spec.tmap_arg, spec.pad_mode, fill, len(fill),
                                   _stream()), 'rua_row_map')
        if prof is not None:
            # algorithmic bytes (BASELINE.md section 3): every live token read once, every destination row
            # written once, plus the int64 metadata the kernel consults
            tokens = min(spec.src.rows, spec.dst.rows) if spec.rg._N is None else min(spec.rg._N, spec.src.rows,
                                                                                      spec.dst.rows)
            meta = 8 * spec.rg.B + (8 * spec.rg.Tp if PACK in (spec.src.layout, spec.dst.layout) else 0)
            _profile_end(prof, 'row_map', tokens * row_bytes + rows * row_bytes + meta)
    return out


class _RowMap(torch.autograd.Function):
    @staticmethod
    def forward(ctx, src: Tensor, spec: MapSpec, fill: bytes):
        ctx.spec = spec
        ctx.src_rows = src.shape[0]
        flat = src.detach()
        if not flat.is_contiguous():
            flat = flat.contiguous()
        return _row_map_raw(flat, spec, fill, tuple(src.shape[1:]), src.dtype, src.device)

    @staticmethod
    def backward(ctx, grad_out: Tensor):
        spec: MapSpec = ctx.spec
        g = grad_out.contiguous()
        if spec.pad_mode in (PAD_WRAP, PAD_ROW0) and ctx.src_rows > 0 and g.shape[0] > 0 and g.dtype in _DTYPES:
            # The forward pass was not injective: last() / segment_last of an EMPTY sequence read a wrapped row
            # (select/last.py:11-13), L / R.roll fill their padding slots with flat row 0 (select/roll.py:19-34) -- one
            # source row feeds several outputs and the inverse map is not a map.  Push the source row numbers through the
            # SAME forward map and sum the gradient rows per source row (stable device sort + one gathered segment-sum
            # launch: deterministic, no atomics); fill = one-past-the-end = a bucket that is dropped.
            rows = ctx.src_rows
            ids = torch.arange(rows, dtype=torch.long, device=g.device)
            where = _row_map_raw(ids, spec, int(rows).to_bytes(8, 'little'), (), torch.long, g.device)
            red, _ = scatter_reduce(g, where, rows + 1, 'sum')
            return red[:rows], None, None
        inv = spec.inverse()
        zero = bytes(g.element_size())
        grad_src = _row_map_raw(g, inv, zero, tuple(g.shape[1:]), g.dtype, g.device)
        return grad_src, None, None


def row_map_mask(src_flat: Tensor, spec: MapSpec, fill_value, zero, one, mask_dtype: torch.dtype):
    """padded (LEFT) destination AND its (B, W) mask from one decode (rua_row_map_mask); None when the fused kernel does
    not apply (narrow rows, gradients wanted) -- the caller then issues the two launches."""
    lib = _lib.load()
    require_cuda(src_flat)
    if src_flat.requires_grad and torch.is_grad_enabled():
        return None
    feat = tuple(src_flat.shape[1:])
    row_bytes = src_flat.element_size()
    for f in feat:
        row_bytes *= f
    rows = spec.dst.rows
    if row_bytes < 128 or rows == 0 or spec.dst.layout != LEFT:
        return None
    flat = src_flat if src_flat.is_contiguous() else src_flat.contiguous()
    out = torch.empty((rows,) + feat, dtype=flat.dtype, device=flat.device)
    mask_out = torch.empty((rows,), dtype=mask_dtype, device=flat.device)
    fill = scalar_bytes(fill_value, flat.dtype)
    z, o = scalar_bytes(zero, mask_dtype), scalar_bytes(one, mask_dtype)
    rg, sd, dd = spec.rg.c_struct(), spec.src.c_struct(), spec.dst.c_struct()
    with _on(flat.device):
        prof = _profile_begin()
        _lib.check(lib.rua_row_map_mask(_ptr(flat), out.data_ptr(), row_bytes, ctypes.byref(rg), ctypes.byref(sd),
                                        ctypes.byref(dd), fill, len(fill), z, o, mask_out.element_size(),
                                        mask_out.data_ptr(), _stream()), 'rua_row_map_mask')
        if prof is not None:
            tokens = min(spec.src.rows, rows) if spec.rg._N is None else min(spec.rg._N, spec.src.rows, rows)
            _profile_end(prof, 'row_map_mask', (tokens + rows) * row_bytes + rows * mask_out.element_size() + 8 * spec.rg.B)
    return out, mask_out


def row_map(src_flat: Tensor, spec: MapSpec, fill_value=0) -> Tensor:
    """src_flat: (rows_src, *feat) contiguous flattened storage of the source layout."""
    require_cuda(src_flat)
    fill = scalar_bytes(fill_value, src_flat.dtype)
    if not (src_flat.requires_grad and torch.is_grad_enabled()):   # no graph to record: skip autograd.Function
        flat = src_flat if src_flat.is_contiguous() else src_flat.contiguous()
        return _row_map_raw(flat, spec, fill, tuple(src_flat.shape[1:]), src_flat.dtype, src_flat.device)
    return _RowMap.apply(src_flat, spec, fill)


# ------------------------------------------------------------------------------------------------
# constructors from lists of tensors (C/L/P/R.new): metadata on the HOST (the lengths are shapes: no device
# sync at all), one upload, one multi-source row-map launch
# ------------------------------------------------------------------------------------------------
HOST_SORT_MAX_B = 1 << 16      # above this the stable sort for P.new runs on the device (K0) instead of numpy


def host_metadata(lengths, with_pack: bool):
    """Pure host side of the constructors: (B, N, T, [len, off(B+1)] + ([sorted, unsorted, batch_sizes, poff(T+1)] if
    with_pack), batch_sizes) as int64 numpy arrays -- the same closed forms the K0 kernels compute on the device
    (stable descending order: ties by ascending index).  No torch, no CUDA: covered by the CPU test-suite."""
    import numpy as np
    lens_np = np.asarray(lengths, dtype=np.int64).reshape(-1)
    b = int(lens_np.size)
    n = int(lens_np.sum()) if b else 0
    t = int(lens_np.max()) if b else 0
    parts = [lens_np, np.concatenate(([0], np.cumsum(lens_np))).astype(np.int64)]
    bs = None
    if with_pack:
        srt = np.argsort(-lens_np, kind='stable').astype(np.int64)
        uns = np.empty_like(srt)
        uns[srt] = np.arange(b, dtype=np.int64)
        bs = (np.bincount(lens_np, minlength=t + 1)[::-1].cumsum()[::-1][1:] if t > 0 else np.zeros(0, np.int64)).astype(np.int64)
        parts += [srt, uns, bs, np.concatenate(([0], np.cumsum(bs))).astype(np.int64)]
    return b, n, t, parts, bs


def ragged_from_host_lengths(lengths, device: torch.device, want_pack: bool, extra_host: Optional[Tensor] = None):
    """Ragged for lengths known on the host (list construction).  Everything -- offsets, N, T and, for small
    batches, the stable descending order, batch_sizes and their prefix sums -- is computed with numpy and
    shipped in ONE pinned H2D copy; nothing is read back.  ``extra_host`` (int64) rides along in the same copy
    (the pointer table of the list kernel) and is returned as a device view."""
    b, n, t, parts, bs = host_metadata(lengths, want_pack and 0 < len(lengths) <= HOST_SORT_MAX_B)
    host_pack = len(parts) > 2
    n_extra = 0 if extra_host is None else extra_host.numel()
    sizes = [p.size for p in parts]
    host = torch.empty(sum(sizes) + n_extra, dtype=torch.long, pin_memory=True)
    view = host.numpy()
    at = 0
    for p in parts:
        view[at:at + p.size] = p
        at += p.size
    if n_extra:
        host[at:] = extra_host
    with _on(device):
        devbuf = host.to(device, non_blocking=True)
    cuts, at = [], 0
    for sz in sizes:
        cuts.append(devbuf[at:at + sz])
        at += sz
    rg = Ragged(device=device, B=b, len=cuts[0], off=cuts[1], _N=n, _T=t)
    rg._keep += [devbuf, host]         # the pinned staging buffer must outlive the asynchronous copy
    if host_pack:
        rg.sorted, rg.unsorted, rg.bs_dev, rg.poff = cuts[2], cuts[3], cuts[4], cuts[5]
        rg.Tp = t
        rg.bs_cpu = torch.from_numpy(bs.copy())
        _cache_put(rg.unsorted, 'pack', rg)
    elif want_pack:
        rg.ensure_pack()
    _cache_put(rg.len, 'len', rg)
    return rg, (devbuf[at:] if n_extra else None)


def _list_row_bytes(t: Tensor) -> int:
    n = t.element_size()
    for f in t.shape[1:]:
        n *= f
    return n


_T_SIZE, _T_PTR, _T_CONTIG, _T_DEV = Tensor.size, Tensor.data_ptr, Tensor.is_contiguous, Tensor.get_device


def _dtype_of(t):
    return t.dtype


def list_plan(tensors):
    """One cheap pass over the list (this is host-bound for thousands of tensors: ~0.5 us per tensor, no per-tensor
    Tensor objects created).  None if the multi-source kernel cannot take it (CPU tensors, mixed dtypes / devices /
    trailing shapes): the caller then goes through torch.cat and gets ATen's promotion rules and error messages."""
    if len(tensors) == 0 or not all(isinstance(t, Tensor) for t in tensors):
        return None
    t0 = tensors[0]
    if not t0.is_cuda or t0.dim() < 1:
        return None
    sizes = list(map(_T_SIZE, tensors))
    feat = sizes[0][1:]
    if len(set(map(_dtype_of, tensors))) != 1 or len(set(map(_T_DEV, tensors))) != 1:
        return None
    if any(sz[1:] != feat for sz in sizes):
        return None
    keep = tensors
    if not all(map(_T_CONTIG, tensors)):
        keep = [t if t.is_contiguous() else t.contiguous() for t in tensors]
    ptrs = list(map(_T_PTR, keep))
    return [sz[0] for sz in sizes], ptrs, tuple(feat), keep


def _list_forward(tensors, layout: int, fill: bytes, plan):
    """-> (data in `layout`, Ragged, destination side)."""
    lib = _lib.load()
    lengths, ptrs, feat, keep = plan
    t0 = tensors[0]
    dev = t0.device
    bits = 0
    for q in ptrs:
        bits |= q
    align = 32
    while bits % align:
        align >>= 1
    rg, ptr_dev = ragged_from_host_lengths(lengths, dev, layout == PACK, torch.tensor(ptrs, dtype=torch.long))
    b, t, n = rg.B, rg._T, rg._N
    if layout in (LEFT, RIGHT):
        side, shape = SideSpec(layout, width=t, rows=b * t), (b, t) + feat
    else:
        side, shape = SideSpec(layout, rows=n), (n,) + feat
    out = torch.empty(shape, dtype=t0.dtype, device=dev)
    row_bytes = _list_row_bytes(t0)
    if out.numel() > 0:
        rgc, d = rg.c_struct(), side.c_struct()
        with _on(dev):
            _lib.check(lib.rua_row_map_list(ptr_dev.data_ptr(), align, out.data_ptr(), row_bytes, ctypes.byref(rgc),
                                            ctypes.byref(d), fill, len(fill), _stream()), 'rua_row_map_list')
    del keep   # contiguous temporaries (if any) are released stream-ordered by the caching allocator
    return out, rg, side


class _ListNew(torch.autograd.Function):
    """list of (len_i, *feat) tensors -> data of a C / L / P / R sequence; gradients flow back to every tensor."""

    @staticmethod
    def forward(ctx, layout: int, fill: bytes, holder: list, plan, *tensors: Tensor):
        out, rg, side = _list_forward(tensors, layout, fill, plan)
        ctx.rg, ctx.side = rg, side
        ctx.lengths = plan[0]
        holder.append(rg)
        return out

    @staticmethod
    def backward(ctx, grad_out: Tensor):
        rg, side = ctx.rg, ctx.side
        g = grad_out.contiguous()
        if side.layout != CAT:   # back to sequence-major rows: one inverse row map
            flat = g.view((side.rows,) + tuple(g.shape[2:] if side.layout in (LEFT, RIGHT) else g.shape[1:]))
            spec = MapSpec(rg=rg, src=side, dst=SideSpec(CAT, rows=rg.N))
            g = _row_map_raw(flat, spec, bytes(g.element_size()), tuple(flat.shape[1:]), g.dtype, g.device)
        return (None, None, None, None) + tuple(g.split(ctx.lengths, dim=0))


def new_from_list(tensors, layout: int, fill_value, plan):
    """-> (data, Ragged) of the list laid out as `layout`; one kernel, no host sync.  plan = list_plan(tensors)."""
    fill = scalar_bytes(fill_value, tensors[0].dtype)
    if torch.is_grad_enabled() and any(t.requires_grad for t in tensors):
        holder = []
        out = _ListNew.apply(layout, fill, holder, plan, *tensors)
        return out, holder[0]
    out, rg, _ = _list_forward(tensors, layout, fill, plan)
    return out, rg


def index_errors(reset: bool = True) -> int:
    """out-of-range indices seen by the gather / scatter / position-key kernels on the current device since the last
    reset (those rows were zero-filled / skipped, never dereferenced).  Synchronises; diagnostics only."""
    lib = _lib.load()
    n = ctypes.c_int64(0)
    _lib.check(lib.rua_index_error_count(ctypes.byref(n), int(reset)), 'rua_index_error_count')
    return int(n.value)


def token_rows(rg: Optional[Ragged], side: 'SideSpec', T: int, batch_ptr: Optional[Tensor], token_ptr: Tensor) -> Tensor:
    """flat storage rows of (batch_ptr, token_ptr) position keys in the layout described by ``side`` (core/get.py:21-82);
    ``batch_ptr=None``: ``token_ptr`` holds flat rows, which are wrapped (negative indices) and bounds-checked."""
    lib = _lib.load()
    if batch_ptr is not None:
        if batch_ptr.shape != token_ptr.shape:
            batch_ptr, token_ptr = torch.broadcast_tensors(batch_ptr, token_ptr)
        b = _i64(batch_ptr)
    t = _i64(token_ptr)
    out = torch.empty(t.shape, dtype=torch.long, device=t.device)
    if out.numel() > 0:
        sd = side.c_struct()
        rgc = rg.c_struct() if batch_ptr is not None else None
        with _on(t.device):
            _lib.check(lib.rua_token_rows(ctypes.byref(rgc) if rgc is not None else None, ctypes.byref(sd), T,
                                          b.data_ptr() if batch_ptr is not None else None, t.data_ptr(), t.numel(),
                                          out.data_ptr(), _stream()), 'rua_token_rows')
    return out


def _gather_rows_raw(flat: Tensor, idx: Tensor) -> Tensor:
    """flat (rows, *feat) contiguous, idx int64 contiguous of any shape -> (idx.numel(), *feat)."""
    lib = _lib.load()
    out = torch.empty((idx.numel(),) + tuple(flat.shape[1:]), dtype=flat.dtype, device=flat.device)
    if out.numel() > 0:
        row_bytes = flat.element_size() * (flat[0].numel() if flat.shape[0] else 0)
        with _on(flat.device):
            _lib.check(lib.rua_gather_rows(flat.data_ptr(), flat.shape[0], idx.data_ptr(), idx.numel(),
                                           row_bytes, out.data_ptr(), _stream()), 'rua_gather_rows')
    return out


def _scatter_rows_raw(dst: Tensor, idx: Tensor, val: Tensor) -> None:
    """dst (rows, *feat) contiguous, idx (n,) int64, val (n, *feat) contiguous: dst[idx[j]] = val[j]."""
    lib = _lib.load()
    if val.numel() == 0:
        return
    row_bytes = dst.element_size() * (dst[0].numel())
    with _on(dst.device):
        _lib.check(lib.rua_scatter_rows(val.data_ptr(), idx.data_ptr(), idx.numel(), row_bytes, dst.data_ptr(),
                                        dst.shape[0], _stream()), 'rua_scatter_rows')


class _GatherRows(torch.autograd.Function):
    @staticmethod
    def forward(ctx, src: Tensor, index: Tensor):
        idx = _i64(index)
        ctx.save_for_backward(idx)
        ctx.src_shape = src.shape
        flat = src.detach().contiguous()
        out = _gather_rows_raw(flat, idx)
        return out.view(tuple(index.shape) + tuple(flat.shape[1:]))

    @staticmethod
    def backward(ctx, grad_out: Tensor):
        (idx,) = ctx.saved_tensors
        rows = ctx.src_shape[0]
        feat = tuple(ctx.src_shape[1:])
        if idx.numel() == 0 or rows == 0:
            return torch.zeros(ctx.src_shape, dtype=grad_out.dtype, device=grad_out.device), None
        # user indices may repeat: the gradient of a row is the SUM over its occurrences.  Native and deterministic:
        # normalise the indices (wrap + bounds; out-of-range ones go to an extra bucket `rows`), stable device sort,
        # then one segment-reduce launch that gathers grad rows in sorted order (no atomics; fp32 accumulation).
        norm = token_rows(None, SideSpec(CAT, rows=rows), 0, None, idx.view(-1))
        g = grad_out.reshape((-1,) + feat)
        if g.dtype in _DTYPES:
            red, _ = scatter_reduce(g if g.is_contiguous() else g.contiguous(), norm, rows + 1, 'sum')
            return red[:rows], None
        grad = torch.zeros(ctx.src_shape, dtype=grad_out.dtype, device=grad_out.device)   # integer / complex grads: ATen
        grad.index_put_((norm.clamp_max(rows - 1),), g, accumulate=True)
        return grad, None


def gather_rows(src: Tensor, index: Tensor) -> Tensor:
    require_cuda(src, index)
    if not (src.requires_grad and torch.is_grad_enabled()):
        flat = src.detach()
        if not flat.is_contiguous():
            flat = flat.contiguous()
        return _gather_rows_raw(flat, _i64(index)).view(tuple(index.shape) + tuple(flat.shape[1:]))
    return _GatherRows.apply(src, index)


class _GatherRowsMulti(torch.autograd.Function):
    """rows ``index`` of the VIRTUAL concatenation of several (rows_k, *feat) tensors -- compose (torchrua/compose.py:33:
    ``torch.cat(data, dim=0)[indices]``) without the concatenation pass: every payload byte moves once."""

    @staticmethod
    def forward(ctx, index: Tensor, *payloads: Tensor):
        out, bases = _gather_rows_multi_raw(index, [p.detach() for p in payloads])
        ctx.save_for_backward(index)
        ctx.bases = bases
        ctx.shapes = [tuple(p.shape) for p in payloads]
        return out

    @staticmethod
    def backward(ctx, grad_out: Tensor):
        (index,) = ctx.saved_tensors
        total = ctx.bases[-1]
        g = grad_out.contiguous()
        feat = tuple(g.shape[1:])
        # compose's index visits every live row exactly once (padding rows of L / R sources: never): one scatter into
        # the concatenated gradient, whose slices are the gradients of the sources (views, no copies)
        cat = torch.zeros((total,) + feat, dtype=g.dtype, device=g.device)
        if index.numel() > 0:
            _scatter_rows_raw(cat, _i64(index).view(-1), g)
        grads = tuple(cat[ctx.bases[k]:ctx.bases[k + 1]].view(shape) for k, shape in enumerate(ctx.shapes))
        return (None,) + grads


def _gather_rows_multi_raw(index: Tensor, payloads):
    lib = _lib.load()
    flats = [p if p.is_contiguous() else p.contiguous() for p in payloads]
    dev = flats[0].device
    feat = tuple(flats[0].shape[1:])
    dtype = flats[0].dtype
    for f in flats:
        if tuple(f.shape[1:]) != feat or f.dtype != dtype or f.device != dev:
            raise RuntimeError('torchrua_b200: compose needs sequences of one dtype, device and feature shape')
    bases = [0]
    for f in flats:
        bases.append(bases[-1] + f.shape[0])
    ptrs = [f.data_ptr() for f in flats]
    bits = 0
    for q in ptrs:
        bits |= q
    align = 32
    while bits % align:
        align >>= 1
    idx = _i64(index).view(-1)
    out = torch.empty((idx.numel(),) + feat, dtype=dtype, device=dev)
    if out.numel() > 0:
        row_bytes = out.element_size()
        for f in feat:
            row_bytes *= f
        k = len(flats)
        table = upload(torch.tensor(ptrs + bases, dtype=torch.long), dev)      # [pointers (k) | bases (k + 1)], one H2D
        with _on(dev):
            _lib.check(lib.rua_gather_rows_multi(table.data_ptr(), table.data_ptr() + 8 * k, k, align, idx.data_ptr(),
                                                 idx.numel(), row_bytes, out.data_ptr(), _stream()),
                       'rua_gather_rows_multi')
    return out, bases


def gather_rows_multi(index: Tensor, payloads) -> Tensor:
    require_cuda(index, *payloads)
    if torch.is_grad_enabled() and any(p.requires_grad for p in payloads):
        return _GatherRowsMulti.apply(index, *payloads)
    return _gather_rows_multi_raw(index, payloads)[0]


def _bump_version(t: Tensor) -> None:
    """a write through the raw pointer is invisible to autograd's and this package's own version checks."""
    torch.autograd.graph.increment_version(t)


def scatter_rows_(dst: Tensor, index: Tensor, value) -> None:
    """dst[index[j]] = value[j] in place, outside autograd (the tracked case is _ScatterRows)."""
    require_cuda(dst, index)
    if not dst.is_contiguous():
        raise RuntimeError('torchrua_b200: in-place scatter needs a contiguous destination')
    idx = _i64(index).view(-1)
    feat = tuple(dst.shape[1:])
    val = torch.as_tensor(value, dtype=dst.dtype, device=dst.device)
    val = val.expand((idx.numel(),) + feat).contiguous()
    _scatter_rows_raw(dst, idx, val)
    _bump_version(dst)


class _ScatterRows(torch.autograd.Function):
    """tracked ``dst[index] = value`` (core/set.py under autograd; ATen's IndexPutBackward0): the destination is modified
    in place (mark_dirty), its gradient is the incoming one with the overwritten rows zeroed, the value's gradient is the
    incoming rows gathered at ``index`` (summed over broadcast dimensions)."""

    @staticmethod
    def forward(ctx, dst: Tensor, index: Tensor, value: Tensor):
        ctx.mark_dirty(dst)
        idx = _i64(index).view(-1)
        feat = tuple(dst.shape[1:])
        ctx.value_shape = tuple(value.shape)
        ctx.save_for_backward(idx)
        val = value.detach().to(dtype=dst.dtype).expand((idx.numel(),) + feat).contiguous()
        _scatter_rows_raw(dst, idx, val)
        return dst

    @staticmethod
    def backward(ctx, grad: Tensor):
        (idx,) = ctx.saved_tensors
        g = grad.contiguous()
        grad_value = grad_dst = None
        if ctx.needs_input_grad[2]:
            grad_value = _gather_rows_raw(g, idx).sum_to_size(ctx.value_shape) if idx.numel() else g.new_zeros(ctx.value_shape)
        if ctx.needs_input_grad[0]:
            grad_dst = g.clone()
            if idx.numel():
                _scatter_rows_raw(grad_dst, idx, g.new_zeros((1,) + tuple(g.shape[1:])).expand((idx.numel(),) + tuple(g.shape[1:])).contiguous())
        return grad_dst, None, grad_value


def scatter_rows_tracked_(dst: Tensor, index: Tensor, value) -> None:
    require_cuda(dst, index)
    if not dst.is_contiguous():
        raise RuntimeError('torchrua_b200: in-place scatter needs a contiguous destination')
    val = value if isinstance(value, Tensor) else torch.as_tensor(value, dtype=dst.dtype, device=dst.device)
    _ScatterRows.apply(dst, index, val)


# ------------------------------------------------------------------------------------------------
# K3: mask / index emit
# ------------------------------------------------------------------------------------------------
def mask(rg: Ragged, width: int, zero, one, dtype: torch.dtype) -> Tensor:
    lib = _lib.load()
    out = torch.empty((rg.B, width), dtype=dtype, device=rg.device)
    if out.numel() == 0:
        return out
    z, o = scalar_bytes(zero, dtype), scalar_bytes(one, dtype)
    with _on(rg.device):
        prof = _profile_begin()
        _lib.check(lib.rua_mask(rg.len.data_ptr(), rg.B, width, z, o, out.element_size(), out.data_ptr(),
                                _stream()), 'rua_mask')
        if prof is not None:
            _profile_end(prof, 'mask', out.numel() * out.element_size() + 8 * rg.B)
    return out


def emit_ptr(off: Tensor, n: int, relabel: Optional[Tensor] = None, want_which=True, want_within=True,
             flat_stride: int = 0, right_align: bool = False):
    lib = _lib.load()
    dev = off.device
    S = off.numel() - 1
    which = torch.empty(n, dtype=torch.long, device=dev) if want_which else None
    within = torch.empty(n, dtype=torch.long, device=dev) if want_within else None
    flat = torch.empty(n, dtype=torch.long, device=dev) if flat_stride else None
    if n > 0:
        with _on(dev):
            prof = _profile_begin()
            _lib.check(lib.rua_emit_ptr(off.data_ptr(), S, n, _ptr(relabel), _ptr(which), _ptr(within), _ptr(flat),
                                        flat_stride, int(right_align), _stream()), 'rua_emit_ptr')
            if prof is not None:
                outs = int(want_which) + int(want_within) + int(bool(flat_stride))
                _profile_end(prof, 'emit_ptr', 8 * n * outs + 8 * S)
    return which, within, flat


# ------------------------------------------------------------------------------------------------
# K4: segment reduce (+ autograd)
# ------------------------------------------------------------------------------------------------
# parity mode (SURVEY.md 8c hazard 2): sum / mean / prod replay torch.segment_reduce's order of operations
# (sequential, one rounding to the storage dtype per step) and match the reference bit for bit
STRICT_REDUCTIONS = False
_STRICT_OPS = (_lib.SUM, _lib.MEAN, _lib.PROD)


class strict_reductions:
    """``with strict_reductions():`` -- segment_sum / segment_mean / segment_prod (and .seg(...) through them)
    return exactly the bits of the reference; the default fast kernels stay within the stated tolerance of it
    (fp32 accumulation, one rounding) and are closer to the true value for 16-bit data.  The prefix scans
    (segment_cumsum / logcumsumexp / cummax / cummin and their layout methods) are not affected: they always
    accumulate in fp32 (fp64 for fp64) with one rounding."""

    def __init__(self, enabled: bool = True):
        self.enabled = enabled

    def __enter__(self):
        global STRICT_REDUCTIONS
        self.prev, STRICT_REDUCTIONS = STRICT_REDUCTIONS, self.enabled
        return self

    def __exit__(self, *exc):
        global STRICT_REDUCTIONS
        STRICT_REDUCTIONS = self.prev
        return False


def _reduce_raw(data: Tensor, off: Tensor, S: int, op: int, rows: Optional[Tensor] = None) -> Tensor:
    """out[s] = reduce(data[off[s]:off[s + 1]]), or with `rows` reduce(data[rows[off[s]:off[s + 1]]]) (the kernel gathers
    the rows; no strict mode)."""
    lib = _lib.load()
    if data.dtype not in _DTYPES:
        if rows is not None:
            raise RuntimeError(f'torchrua_b200: scatter reductions support float16/bfloat16/float32/float64, got {data.dtype}')
        raise RuntimeError(f'torchrua_b200: segment reductions support float16/bfloat16/float32/float64, got '
                           f'{data.dtype} (the reference rejects integer data too: "_segment_reduce" not '
                           f'implemented for Long)')
    N = data.shape[0] if rows is None else rows.numel()
    feat = tuple(data.shape[1:])
    H = 1
    for f in feat:
        H *= f
    out = torch.empty((S,) + feat, dtype=data.dtype, device=data.device)
    if out.numel() == 0:
        return out
    dt = _DTYPES[data.dtype]
    if rows is None and STRICT_REDUCTIONS and op in _STRICT_OPS:
        with _on(data.device):
            _lib.check(lib.rua_segment_reduce_strict(_ptr(data), off.data_ptr(), N, S, H, dt, op, out.data_ptr(),
                                                     _stream()), 'rua_segment_reduce_strict')
        return out
    with _on(data.device):
        nbytes = lib.rua_segment_reduce_workspace_bytes(N, S, H, dt, op)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=data.device)
        prof = _profile_begin()
        if rows is None:
            _lib.check(lib.rua_segment_reduce(_ptr(data), off.data_ptr(), N, S, H, dt, op, out.data_ptr(),
                                              ws.data_ptr(), nbytes, _stream()), 'rua_segment_reduce')
        else:
            _lib.check(lib.rua_segment_reduce_gather(_ptr(data), rows.data_ptr(), off.data_ptr(), N, S, H, dt, op,
                                                     out.data_ptr(), ws.data_ptr(), nbytes, _stream()),
                       'rua_segment_reduce_gather')
        if prof is not None:
            if rows is None:
                _profile_end(prof, 'segment_reduce', (N + S) * H * data.element_size() + 8 * S)
            else:
                _profile_end(prof, 'segment_reduce_gather', (N + S) * H * data.element_size() + 8 * (S + N))
    return out


def _reduce_backward_raw(grad_out: Tensor, out: Tensor, data: Tensor, off: Tensor, S: int, op: int,
                         grad: Tensor) -> None:
    """grad (the shape of data, at least one element) = gradient of out = _reduce_raw(data, off, S, op)."""
    lib = _lib.load()
    N = data.shape[0]
    H = data[0].numel()
    dt = _DTYPES[data.dtype]
    with _on(data.device):
        nbytes = lib.rua_segment_reduce_backward_workspace_bytes(N, S, H, dt, op)
        ws = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=data.device)
        _lib.check(lib.rua_segment_reduce_backward(grad_out.data_ptr(), out.data_ptr(), data.data_ptr(), off.data_ptr(),
                                                   N, S, H, dt, op, grad.data_ptr(), ws.data_ptr(), nbytes, _stream()),
                   'rua_segment_reduce_backward')


class _SegmentReduce(torch.autograd.Function):
    @staticmethod
    def forward(ctx, data: Tensor, off: Tensor, S: int, op: int):
        flat = data.detach()
        if not flat.is_contiguous():
            flat = flat.contiguous()
        out = _reduce_raw(flat, off, S, op)
        ctx.op = op
        ctx.S = S
        ctx.save_for_backward(flat, off, out)
        return out

    @staticmethod
    def backward(ctx, grad_out: Tensor):
        data, off, out = ctx.saved_tensors
        grad = torch.empty_like(data)
        if grad.numel() > 0:
            _reduce_backward_raw(grad_out.contiguous(), out, data, off, ctx.S, ctx.op, grad)
        return grad, None, None, None


def segment_reduce(data: Tensor, segment_sizes: Tensor, op: str) -> Tensor:
    require_cuda(data, segment_sizes)
    rg = ragged_from_lengths(segment_sizes)
    if not (data.requires_grad and torch.is_grad_enabled()):
        return _reduce_raw(data if data.is_contiguous() else data.contiguous(), rg.off, rg.B, _OPS[op])
    return _SegmentReduce.apply(data, rg.off, rg.B, _OPS[op])


# ------------------------------------------------------------------------------------------------
# K6: per-sequence prefix scans (+ autograd)
# ------------------------------------------------------------------------------------------------
_SCAN_OPS = {'sum': _lib.SCAN_SUM, 'logsumexp': _lib.SCAN_LOGSUMEXP, 'max': _lib.SCAN_MAX, 'min': _lib.SCAN_MIN}


def _scan_check(data: Tensor) -> None:
    if data.dtype not in _DTYPES:
        raise RuntimeError(f'torchrua_b200: segment scans support float16/bfloat16/float32/float64, got {data.dtype}')


def _scan_raw(data: Tensor, rg: Ragged, side: SideSpec, op: int, reverse: bool):
    """(out, idx or None) with out laid out like data; data: (side.rows, *feat) contiguous."""
    lib = _lib.load()
    H = data[0].numel() if data.shape[0] else 0
    out = torch.empty_like(data)
    idx = torch.empty(data.shape, dtype=torch.long, device=data.device) if op in (_lib.SCAN_MAX, _lib.SCAN_MIN) else None
    if out.numel() == 0:
        return out, idx
    dt = _DTYPES[data.dtype]
    c_rg, c_side = rg.c_struct(), side.c_struct()
    with _on(data.device):
        nbytes = lib.rua_segment_scan_workspace_bytes(side.rows, H, dt, op, 0)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=data.device)
        prof = _profile_begin()
        _lib.check(lib.rua_segment_scan(data.data_ptr(), out.data_ptr(), _ptr(idx), H, dt, op, int(reverse),
                                        ctypes.byref(c_rg), ctypes.byref(c_side), ws.data_ptr(), nbytes, _stream()),
                   'rua_segment_scan')
        if prof is not None:
            # every row read once and written once (+ the int64 indices of max / min) + the metadata consulted
            nb = 2 * data.numel() * data.element_size() + (8 * data.numel() if idx is not None else 0)
            _profile_end(prof, 'segment_scan', nb + 8 * rg.B + (8 * (rg.Tp + rg.B) if side.layout == PACK else 0))
    return out, idx


def _scan_backward_raw(g: Tensor, x: Optional[Tensor], y: Optional[Tensor], idx: Optional[Tensor], rg: Ragged,
                       side: SideSpec, op: int, reverse: bool) -> Tensor:
    lib = _lib.load()
    g = g.contiguous()
    grad = torch.empty_like(g)   # every row is written by the kernel (non-token rows pass grad_out through)
    if grad.numel() == 0:
        return grad
    H = g[0].numel()
    dt = _DTYPES[g.dtype]
    c_rg, c_side = rg.c_struct(), side.c_struct()
    with _on(g.device):
        nbytes = lib.rua_segment_scan_workspace_bytes(side.rows, H, dt, op, 1)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=g.device)
        prof = _profile_begin()
        _lib.check(lib.rua_segment_scan_backward(g.data_ptr(), _ptr(x), _ptr(y), _ptr(idx), grad.data_ptr(), H, dt, op,
                                                 int(reverse), ctypes.byref(c_rg), ctypes.byref(c_side), ws.data_ptr(),
                                                 nbytes, _stream()), 'rua_segment_scan_backward')
        if prof is not None:
            nb = g.numel() * g.element_size() * (4 if op == _lib.SCAN_LOGSUMEXP else 2)
            _profile_end(prof, 'segment_scan_backward', nb + (8 * g.numel() if idx is not None else 0) + 8 * rg.B)
    return grad


class _ScanSum(torch.autograd.Function):
    @staticmethod
    def forward(ctx, data: Tensor, rg: Ragged, side: SideSpec, reverse: bool):
        ctx.meta = (rg, side, reverse)
        return _scan_raw(data.detach().contiguous(), rg, side, _lib.SCAN_SUM, reverse)[0]

    @staticmethod
    def backward(ctx, grad_out: Tensor):
        rg, side, reverse = ctx.meta
        # the gradient of a prefix sum is the suffix sum: the differentiable call, so double backward works
        return segment_scan(grad_out, rg, side, 'sum', not reverse)[0], None, None, None


class _ScanLogSumExp(torch.autograd.Function):
    @staticmethod
    def forward(ctx, data: Tensor, rg: Ragged, side: SideSpec, reverse: bool):
        x = data.detach().contiguous()
        y = _scan_raw(x, rg, side, _lib.SCAN_LOGSUMEXP, reverse)[0]
        ctx.meta = (rg, side, reverse)
        ctx.save_for_backward(x, y)
        return y

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_out: Tensor):
        rg, side, reverse = ctx.meta
        x, y = ctx.saved_tensors
        return _scan_backward_raw(grad_out, x, y, None, rg, side, _lib.SCAN_LOGSUMEXP, reverse), None, None, None


class _ScanExtreme(torch.autograd.Function):
    @staticmethod
    def forward(ctx, data: Tensor, rg: Ragged, side: SideSpec, op: int, reverse: bool):
        out, idx = _scan_raw(data.detach().contiguous(), rg, side, op, reverse)
        ctx.meta = (rg, side, op, reverse)
        ctx.save_for_backward(idx)
        ctx.mark_non_differentiable(idx)
        return out, idx

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_out: Tensor, _grad_idx):
        rg, side, op, reverse = ctx.meta
        idx, = ctx.saved_tensors
        return _scan_backward_raw(grad_out, None, None, idx, rg, side, op, reverse), None, None, None, None


def segment_scan(data: Tensor, rg: Ragged, side: SideSpec, op: str, reverse: bool):
    """per-sequence inclusive scan of the flattened storage ``data`` (side.rows, *feat) -> (out, idx or None)."""
    _scan_check(data)
    require_cuda(data)
    code = _SCAN_OPS[op]
    grad = data.requires_grad and torch.is_grad_enabled()
    if not grad:
        return _scan_raw(data if data.is_contiguous() else data.contiguous(), rg, side, code, reverse)
    if code == _lib.SCAN_SUM:
        return _ScanSum.apply(data, rg, side, reverse), None
    if code == _lib.SCAN_LOGSUMEXP:
        return _ScanLogSumExp.apply(data, rg, side, reverse), None
    return _ScanExtreme.apply(data, rg, side, code, reverse)


def linrec_check(data: Tensor, gate: Tensor, initial: Optional[Tensor], B: int, feat: Tuple[int, ...]) -> None:
    """validate a linear recurrence over rows with features ``feat`` of B sequences, before any device work."""
    if data.dtype not in _DTYPES:
        raise RuntimeError(f'torchrua_b200: linear_recurrence supports float16/bfloat16/float32/float64, got {data.dtype}')
    for name, t in (('gate', gate), ('initial', initial)):
        if t is not None and t.dtype != data.dtype:
            raise RuntimeError(f'torchrua_b200: linear_recurrence {name} has dtype {t.dtype}, the input {data.dtype}')
    if tuple(gate.shape) != tuple(data.shape):
        raise ValueError(f'torchrua_b200: linear_recurrence gate must have the shape of the input {tuple(data.shape)}, '
                         f'got {tuple(gate.shape)}')
    if initial is not None and tuple(initial.shape) != (B,) + tuple(feat):
        raise ValueError(f'torchrua_b200: linear_recurrence initial must be (B, *feat) = {(B,) + tuple(feat)}, '
                         f'got {tuple(initial.shape)}')
    require_cuda(data, gate, initial)


def _linrec_raw(data: Tensor, gate: Tensor, h0: Optional[Tensor], rg: Ragged, side: SideSpec, reverse: bool) -> Tensor:
    """y laid out like data; data, gate (side.rows, *feat) and h0 (B, *feat) or None, all contiguous."""
    lib = _lib.load()
    out = torch.empty_like(data)
    if out.numel() == 0:
        return out
    H = data[0].numel()
    dt = _DTYPES[data.dtype]
    c_rg, c_side = rg.c_struct(), side.c_struct()
    with _on(data.device):
        nbytes = lib.rua_segment_linrec_workspace_bytes(side.rows, H, dt, 0)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=data.device)
        prof = _profile_begin()
        _lib.check(lib.rua_segment_linrec(data.data_ptr(), gate.data_ptr(), _ptr(h0), out.data_ptr(), H, dt, int(reverse),
                                          ctypes.byref(c_rg), ctypes.byref(c_side), ws.data_ptr(), nbytes, _stream()),
                   'rua_segment_linrec')
        if prof is not None:
            # x and the gate read once, y written once + the initial states + the metadata consulted
            nb = 3 * data.numel() * data.element_size() + (h0.numel() * h0.element_size() if h0 is not None else 0)
            _profile_end(prof, 'segment_linrec', nb + 8 * rg.B + (8 * (rg.Tp + rg.B) if side.layout == PACK else 0))
    return out


def _linrec_backward_raw(g: Tensor, gate: Tensor, h0: Optional[Tensor], y: Optional[Tensor], rg: Ragged, side: SideSpec,
                         reverse: bool, want_x: bool, want_gate: bool, want_h0: bool):
    """(grad_x, grad_gate, grad_h0), None where not wanted; g, gate, y (side.rows, *feat) contiguous, y needed for
    grad_gate only."""
    lib = _lib.load()
    gx = torch.empty_like(g) if want_x else None
    gg = torch.empty_like(g) if want_gate else None
    gh = torch.empty((rg.B,) + tuple(g.shape[1:]), dtype=g.dtype, device=g.device) if want_h0 else None
    H = int(np.prod(g.shape[1:]))
    if not (want_x or want_gate or want_h0) or H == 0:
        return gx, gg, gh
    dt = _DTYPES[g.dtype]
    c_rg, c_side = rg.c_struct(), side.c_struct()
    with _on(g.device):
        nbytes = lib.rua_segment_linrec_workspace_bytes(side.rows, H, dt, 1)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=g.device)
        prof = _profile_begin()
        _lib.check(lib.rua_segment_linrec_backward(g.data_ptr(), gate.data_ptr(), _ptr(h0), _ptr(y) if want_gate else None,
                                                   _ptr(gx), _ptr(gg), _ptr(gh), H, dt, int(reverse), ctypes.byref(c_rg),
                                                   ctypes.byref(c_side), ws.data_ptr() if nbytes else None, nbytes,
                                                   _stream()), 'rua_segment_linrec_backward')
        if prof is not None:
            # grad_out, the gate and y read once, grad_x and grad_gate written once
            e = g.element_size()
            nb = g.numel() * e * (2 + 2 * want_gate + want_x) + (gh.numel() * e if gh is not None else 0)
            _profile_end(prof, 'segment_linrec_backward', nb + 8 * rg.B + (8 * (rg.Tp + rg.B) if side.layout == PACK else 0))
    return gx, gg, gh


class _LinearRecurrence(torch.autograd.Function):
    """once-differentiable: the backward is a native kernel, double backward is not supported."""

    @staticmethod
    def forward(ctx, data: Tensor, gate: Tensor, initial: Optional[Tensor], rg: Ragged, side: SideSpec, reverse: bool):
        x = data.detach().contiguous()
        a = gate.detach().contiguous()
        h0 = None if initial is None else initial.detach().contiguous()
        y = _linrec_raw(x, a, h0, rg, side, reverse)
        ctx.meta = (rg, side, reverse)
        ctx.save_for_backward(a, h0, y if ctx.needs_input_grad[1] else None)   # y only feeds grad_gate
        return y

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_out: Tensor):
        rg, side, reverse = ctx.meta
        a, h0, y = ctx.saved_tensors
        need = ctx.needs_input_grad
        gx, gg, gh = _linrec_backward_raw(grad_out.contiguous(), a, h0, y, rg, side, reverse, need[0], need[1],
                                          need[2] and h0 is not None)
        return gx, gg, gh, None, None, None


def linear_recurrence(data: Tensor, gate: Tensor, initial: Optional[Tensor], rg: Ragged, side: SideSpec,
                      reverse: bool) -> Tensor:
    """per-sequence h_t = gate_t * h_(t-1) + x_t over the flattened storage ``data`` (side.rows, *feat); gate like data,
    initial (B, *feat) or None; checked by the caller (linrec_check)."""
    grad = torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in (data, gate, initial))
    if grad:
        return _LinearRecurrence.apply(data, gate, initial, rg, side, reverse)
    return _linrec_raw(data.contiguous(), gate.contiguous(), None if initial is None else initial.contiguous(), rg, side,
                       reverse)


# ------------------------------------------------------------------------------------------------
# K8: per-sequence depthwise 1-D convolution (+ autograd)
# ------------------------------------------------------------------------------------------------
CONV_MAX_K = 32


def conv_check(data: Tensor, weight: Tensor, bias: Optional[Tensor], feat: Tuple[int, ...], padding) -> int:
    """validate a depthwise convolution of rows with features ``feat`` -> pad (positions before the current token)."""
    if data.dtype not in _DTYPES:
        raise RuntimeError(f'torchrua_b200: depthwise_conv1d supports float16/bfloat16/float32/float64, got {data.dtype}')
    for name, t in (('weight', weight), ('bias', bias)):
        if t is not None and t.dtype != data.dtype:
            raise RuntimeError(f'torchrua_b200: depthwise_conv1d {name} has dtype {t.dtype}, the input {data.dtype}')
    if weight.dim() != len(feat) + 1 or tuple(weight.shape[:-1]) != tuple(feat):
        raise ValueError(f'torchrua_b200: depthwise_conv1d weight must be (*feat, K) = {tuple(feat)} + (K,), '
                         f'got {tuple(weight.shape)}')
    K = weight.shape[-1]
    if not 1 <= K <= CONV_MAX_K:
        raise ValueError(f'torchrua_b200: depthwise_conv1d supports kernel sizes 1..{CONV_MAX_K}, got {K}')
    if bias is not None and tuple(bias.shape) != tuple(feat):
        raise ValueError(f'torchrua_b200: depthwise_conv1d bias must be {tuple(feat)}, got {tuple(bias.shape)}')
    if padding == 'causal':
        padding = K - 1
    elif padding == 'same':
        padding = (K - 1) // 2
    elif isinstance(padding, bool) or not isinstance(padding, int) or not 0 <= padding <= K - 1:
        raise ValueError(f"torchrua_b200: depthwise_conv1d padding must be 'causal', 'same' or an int in [0, {K - 1}], "
                         f'got {padding!r}')
    require_cuda(data, weight, bias)
    return padding


def _conv_raw(data: Tensor, weight: Tensor, bias: Optional[Tensor], pad: int, rg: Ragged, side: SideSpec) -> Tensor:
    """y laid out like data; data (side.rows, *feat), weight (H, K), bias (H,) or None, all contiguous."""
    lib = _lib.load()
    out = torch.empty_like(data)
    if out.numel() == 0:
        return out
    H, K = weight.shape
    dt = _DTYPES[data.dtype]
    c_rg, c_side = rg.c_struct(), side.c_struct()
    with _on(data.device):
        prof = _profile_begin()
        _lib.check(lib.rua_segment_conv(data.data_ptr(), weight.data_ptr(), _ptr(bias), out.data_ptr(), H, dt, K, pad,
                                        ctypes.byref(c_rg), ctypes.byref(c_side), None, 0, _stream()), 'rua_segment_conv')
        if prof is not None:
            # every row read once and written once + the taps (and bias) + the metadata consulted
            e = data.element_size()
            nb = 2 * data.numel() * e + (K + (bias is not None)) * H * e
            _profile_end(prof, 'segment_conv', nb + 8 * rg.B + (8 * (rg.Tp + rg.B) if side.layout == PACK else 0))
    return out


def _conv_backward_raw(g: Tensor, x: Tensor, weight: Tensor, pad: int, rg: Ragged, side: SideSpec, want_in: bool,
                       want_w: bool, want_b: bool):
    """(grad_in, grad_weight, grad_bias), None where not wanted; g, x (side.rows, *feat) contiguous."""
    lib = _lib.load()
    H, K = weight.shape
    gi = torch.empty_like(g) if want_in else None
    gw = torch.empty_like(weight) if want_w else None
    gb = torch.empty(H, dtype=g.dtype, device=g.device) if want_b else None
    if g.numel() == 0:
        if gw is not None:
            gw.zero_()
        if gb is not None:
            gb.zero_()
        return gi, gw, gb
    dt = _DTYPES[g.dtype]
    c_rg, c_side = rg.c_struct(), side.c_struct()
    with _on(g.device):
        nbytes = lib.rua_segment_conv_workspace_bytes(side.rows, H, K, dt, 1) if (want_w or want_b) else 0
        ws = torch.empty(nbytes, dtype=torch.uint8, device=g.device)
        prof = _profile_begin()
        _lib.check(lib.rua_segment_conv_backward(g.data_ptr(), _ptr(x) if want_w else None, weight.data_ptr(), _ptr(gi),
                                                 _ptr(gw), _ptr(gb), H, dt, K, pad, ctypes.byref(c_rg),
                                                 ctypes.byref(c_side), ws.data_ptr() if nbytes else None, nbytes,
                                                 _stream()), 'rua_segment_conv_backward')
        if prof is not None:
            # grad_out read once, x read once (grad_weight), grad_in written once + taps and their gradients
            e = g.element_size()
            nb = g.numel() * e * (1 + want_w + want_in) + (2 * K + 1) * H * e
            _profile_end(prof, 'segment_conv_backward', nb + 8 * rg.B + (8 * (rg.Tp + rg.B) if side.layout == PACK else 0))
    return gi, gw, gb


class _SegmentConv(torch.autograd.Function):
    """once-differentiable: the backward is a native kernel, double backward is not supported."""

    @staticmethod
    def forward(ctx, data: Tensor, weight: Tensor, bias: Optional[Tensor], pad: int, rg: Ragged, side: SideSpec):
        x = data.detach().contiguous()
        w = weight.detach().reshape(-1, weight.shape[-1]).contiguous()
        b = None if bias is None else bias.detach().reshape(-1).contiguous()
        ctx.meta = (pad, rg, side, weight.shape, None if bias is None else bias.shape)
        ctx.save_for_backward(x if ctx.needs_input_grad[1] else None, w)   # x only feeds grad_weight
        return _conv_raw(x, w, b, pad, rg, side)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_out: Tensor):
        pad, rg, side, wshape, bshape = ctx.meta
        x, w = ctx.saved_tensors
        need = ctx.needs_input_grad
        gi, gw, gb = _conv_backward_raw(grad_out.contiguous(), x, w, pad, rg, side, need[0], need[1],
                                        need[2] and bshape is not None)
        return (gi, None if gw is None else gw.view(wshape), None if gb is None else gb.view(bshape),
                None, None, None)


def segment_conv(data: Tensor, weight: Tensor, bias: Optional[Tensor], padding, rg: Ragged, side: SideSpec) -> Tensor:
    """per-sequence depthwise convolution of the flattened storage ``data`` (side.rows, *feat); weight (*feat, K)."""
    pad = conv_check(data, weight, bias, tuple(data.shape[1:]), padding)
    grad = torch.is_grad_enabled() and (data.requires_grad or weight.requires_grad or
                                        (bias is not None and bias.requires_grad))
    if grad:
        return _SegmentConv.apply(data, weight, bias, pad, rg, side)
    w = weight.reshape(-1, weight.shape[-1]).contiguous()
    b = None if bias is None else bias.reshape(-1).contiguous()
    return _conv_raw(data if data.is_contiguous() else data.contiguous(), w, b, pad, rg, side)


# ------------------------------------------------------------------------------------------------
# K9: per-sequence linear-chain CRF (+ autograd)
# ------------------------------------------------------------------------------------------------
CRF_MAX_K = 64


def crf_check(emissions: Tensor, transitions: Tensor, start: Optional[Tensor], end: Optional[Tensor], lead: int,
              tags: Optional[Tensor] = None) -> int:
    """validate a CRF over emissions with ``lead`` row dimensions and one tag dimension -> K, before any device work;
    ``tags`` must be int64 and shaped like the row dimensions."""
    if emissions.dtype not in _DTYPES:
        raise RuntimeError(f'torchrua_b200: crf supports float16/bfloat16/float32/float64 emissions, got {emissions.dtype}')
    if emissions.dim() != lead + 1:
        raise ValueError(f'torchrua_b200: crf emissions must have {lead} row dimension(s) and one tag dimension, '
                         f'got shape {tuple(emissions.shape)}')
    K = emissions.shape[-1]
    if not 1 <= K <= CRF_MAX_K:
        raise ValueError(f'torchrua_b200: crf supports 1..{CRF_MAX_K} tags, got {K}')
    for name, t in (('transitions', transitions), ('start', start), ('end', end)):
        if t is not None and t.dtype != emissions.dtype:
            raise RuntimeError(f'torchrua_b200: crf {name} has dtype {t.dtype}, the emissions {emissions.dtype}')
    if tuple(transitions.shape) != (K, K):
        raise ValueError(f'torchrua_b200: crf transitions must be (K, K) = {(K, K)}, got {tuple(transitions.shape)}')
    for name, t in (('start', start), ('end', end)):
        if t is not None and tuple(t.shape) != (K,):
            raise ValueError(f'torchrua_b200: crf {name} must be (K,) = {(K,)}, got {tuple(t.shape)}')
    if tags is not None:
        if tags.dtype != torch.long:
            raise RuntimeError(f'torchrua_b200: crf tags must be int64, got {tags.dtype}')
        if tuple(tags.shape) != tuple(emissions.shape[:-1]):
            raise ValueError(f'torchrua_b200: crf tags must have the shape {tuple(emissions.shape[:-1])} of the emission '
                             f'rows, got {tuple(tags.shape)}')
    require_cuda(emissions, transitions, start, end, tags)
    return K


def _crf_acc_dtype(dtype: torch.dtype) -> torch.dtype:
    return torch.float64 if dtype == torch.float64 else torch.float32


def _crf_forward_raw(x: Tensor, tags: Optional[Tensor], W: Tensor, start: Optional[Tensor], end: Optional[Tensor],
                     rg: Ragged, side: SideSpec, keep_state: bool):
    """(log_z, score or None, state or None); x (side.rows, K), tags (side.rows,) or None, all contiguous."""
    lib = _lib.load()
    K = W.shape[0]
    dt = _DTYPES[x.dtype]
    acc = _crf_acc_dtype(x.dtype)
    log_z = torch.empty(rg.B, dtype=acc, device=x.device)
    score = torch.empty(rg.B, dtype=acc, device=x.device) if tags is not None else None
    state = None
    if keep_state:
        state = torch.empty(lib.rua_crf_state_bytes(side.rows, K, dt), dtype=torch.uint8, device=x.device)
    if rg.B == 0:
        return log_z, score, state
    c_rg, c_side = rg.c_struct(), side.c_struct()
    with _on(x.device):
        prof = _profile_begin()
        _lib.check(lib.rua_crf_forward(x.data_ptr(), _ptr(tags), W.data_ptr(), _ptr(start), _ptr(end), log_z.data_ptr(),
                                       _ptr(score), _ptr(state) if state is not None and state.numel() else None, K, dt,
                                       ctypes.byref(c_rg), ctypes.byref(c_side), None, 0, _stream()), 'rua_crf_forward')
        if prof is not None:
            nb = x.numel() * x.element_size() + (state.numel() if state is not None else 0)
            _profile_end(prof, 'crf_forward', nb + 8 * rg.B + (8 * (rg.Tp + rg.B) if side.layout == PACK else 0))
    return log_z, score, state


def _crf_backward_raw(g_z: Tensor, g_s: Optional[Tensor], x: Tensor, tags: Optional[Tensor], W: Tensor,
                      end: Optional[Tensor], state: Tensor, log_z: Tensor, rg: Ragged, side: SideSpec, want_x: bool,
                      want_w: bool, want_start: bool, want_end: bool):
    """(grad_x, grad_W, grad_start, grad_end), None where not wanted; every input contiguous."""
    lib = _lib.load()
    K = W.shape[0]
    dt = _DTYPES[x.dtype]
    gx = torch.empty_like(x) if want_x else None
    gw = torch.empty_like(W) if want_w else None
    gst = torch.empty(K, dtype=x.dtype, device=x.device) if want_start else None
    gen = torch.empty(K, dtype=x.dtype, device=x.device) if want_end else None
    if not (want_x or want_w or want_start or want_end):
        return gx, gw, gst, gen
    c_rg, c_side = rg.c_struct(), side.c_struct()
    with _on(x.device):
        nbytes = lib.rua_crf_workspace_bytes(side.rows, K, dt, _lib.CRF_BACKWARD) if (want_w or want_start or want_end) else 0
        ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
        prof = _profile_begin()
        _lib.check(lib.rua_crf_backward(g_z.data_ptr(), _ptr(g_s), x.data_ptr(), _ptr(tags), W.data_ptr(), None, _ptr(end),
                                        _ptr(state) if state.numel() else None, log_z.data_ptr(), _ptr(gx), _ptr(gw),
                                        _ptr(gst), _ptr(gen), K, dt, ctypes.byref(c_rg), ctypes.byref(c_side),
                                        ws.data_ptr() if nbytes else None, nbytes, _stream()), 'rua_crf_backward')
        if prof is not None:
            nb = x.numel() * x.element_size() * (1 + want_x) + state.numel()
            _profile_end(prof, 'crf_backward', nb + 8 * rg.B + (8 * (rg.Tp + rg.B) if side.layout == PACK else 0))
    return gx, gw, gst, gen


class _SegmentCrf(torch.autograd.Function):
    """log Z (tags is None) or score(tags) - log Z per sequence.  Once-differentiable: the backward is a native kernel,
    double backward is not supported."""

    @staticmethod
    def forward(ctx, x: Tensor, W: Tensor, start: Optional[Tensor], end: Optional[Tensor], tags: Optional[Tensor],
                rg: Ragged, side: SideSpec):
        xs = x.detach().contiguous()
        Ws = W.detach().contiguous()
        ss = None if start is None else start.detach().contiguous()
        es = None if end is None else end.detach().contiguous()
        keep = any(ctx.needs_input_grad[:4])
        log_z, score, state = _crf_forward_raw(xs, tags, Ws, ss, es, rg, side, keep)
        ctx.meta = (rg, side, start is not None, end is not None)
        if keep:
            ctx.save_for_backward(xs, tags, Ws, es, state, log_z)
        return log_z if tags is None else score - log_z

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g: Tensor):
        rg, side, has_start, has_end = ctx.meta
        x, tags, W, end, state, log_z = ctx.saved_tensors
        need = ctx.needs_input_grad
        g = g.contiguous()
        g_z, g_s = (g, None) if tags is None else (-g, g)
        gx, gw, gst, gen = _crf_backward_raw(g_z, g_s, x, tags, W, end, state, log_z, rg, side, need[0], need[1],
                                             need[2] and has_start, need[3] and has_end)
        return gx, gw, gst, gen, None, None, None


def segment_crf(emissions: Tensor, tags: Optional[Tensor], transitions: Tensor, start: Optional[Tensor],
                end: Optional[Tensor], rg: Ragged, side: SideSpec) -> Tensor:
    """log Z (tags None) or the log-likelihood of ``tags`` per sequence over the flattened storage ``emissions``
    (side.rows, K), tags (side.rows,); checked by the caller (crf_check); ``rg`` has its pack side."""
    grad = torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in (emissions, transitions, start, end))
    tags = None if tags is None else tags.contiguous()
    if grad:
        return _SegmentCrf.apply(emissions, transitions, start, end, tags, rg, side)
    log_z, score, _ = _crf_forward_raw(emissions.contiguous(), tags, transitions.contiguous(),
                                       None if start is None else start.contiguous(),
                                       None if end is None else end.contiguous(), rg, side, False)
    return log_z if tags is None else score - log_z


def crf_decode(emissions: Tensor, transitions: Tensor, start: Optional[Tensor], end: Optional[Tensor], rg: Ragged,
               side: SideSpec) -> Tuple[Tensor, Tensor]:
    """(tags (side.rows,) int64 with -1 at rows that hold no token, best score (B,)); no gradient."""
    lib = _lib.load()
    x = emissions.detach().contiguous()
    W, start, end = (None if t is None else t.detach().contiguous() for t in (transitions, start, end))
    K = x.shape[-1]
    dt = _DTYPES[x.dtype]
    tags = torch.empty(side.rows, dtype=torch.long, device=x.device)
    best = torch.empty(rg.B, dtype=_crf_acc_dtype(x.dtype), device=x.device)
    if rg.B == 0 and side.rows == 0:
        return tags, best
    c_rg, c_side = rg.c_struct(), side.c_struct()
    with _on(x.device):
        nbytes = lib.rua_crf_workspace_bytes(side.rows, K, dt, _lib.CRF_DECODE)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
        prof = _profile_begin()
        _lib.check(lib.rua_crf_decode(x.data_ptr(), W.data_ptr(), _ptr(start), _ptr(end), tags.data_ptr(), best.data_ptr(),
                                      K, dt, ctypes.byref(c_rg), ctypes.byref(c_side), ws.data_ptr() if nbytes else None,
                                      nbytes, _stream()), 'rua_crf_decode')
        if prof is not None:
            nb = x.numel() * x.element_size() + 9 * side.rows + 2 * side.rows * K
            _profile_end(prof, 'crf_decode', nb + 8 * rg.B + (8 * (rg.Tp + rg.B) if side.layout == PACK else 0))
    return tags, best


# ------------------------------------------------------------------------------------------------
# K10: per-sequence selective state-space scan (+ autograd)
# ------------------------------------------------------------------------------------------------
SSM_MAX_N = 16


def ssm_check(data: Tensor, delta: Tensor, A: Tensor, Bm: Tensor, Cm: Tensor, initial: Optional[Tensor], B: int,
              lead: int) -> Tuple[Tuple[int, ...], int]:
    """validate a selective scan over ``data`` with ``lead`` row dimensions -> (feat, N), before any device work."""
    if data.dtype not in _DTYPES:
        raise RuntimeError(f'torchrua_b200: selective_scan supports float16/bfloat16/float32/float64, got {data.dtype}')
    acc = _crf_acc_dtype(data.dtype)
    for name, t, want in (('delta', delta, data.dtype), ('B', Bm, data.dtype), ('C', Cm, data.dtype), ('A', A, acc),
                          ('initial', initial, acc)):
        if t is not None and t.dtype != want:
            raise RuntimeError(f'torchrua_b200: selective_scan {name} must have dtype {want} for a {data.dtype} input, '
                               f'got {t.dtype}')
    if data.dim() < lead:
        raise ValueError(f'torchrua_b200: selective_scan input must have {lead} row dimension(s), '
                         f'got shape {tuple(data.shape)}')
    rows, feat = tuple(data.shape[:lead]), tuple(data.shape[lead:])
    if tuple(delta.shape) != tuple(data.shape):
        raise ValueError(f'torchrua_b200: selective_scan delta must have the shape of the input {tuple(data.shape)}, '
                         f'got {tuple(delta.shape)}')
    if Bm.dim() != lead + 1 or tuple(Bm.shape[:lead]) != rows:
        raise ValueError(f'torchrua_b200: selective_scan B must be {rows} + (N,), got {tuple(Bm.shape)}')
    N = Bm.shape[-1]
    if not 1 <= N <= SSM_MAX_N:
        raise ValueError(f'torchrua_b200: selective_scan supports state sizes 1..{SSM_MAX_N}, got {N}')
    if tuple(Cm.shape) != tuple(Bm.shape):
        raise ValueError(f'torchrua_b200: selective_scan C must have the shape of B {tuple(Bm.shape)}, '
                         f'got {tuple(Cm.shape)}')
    if tuple(A.shape) != feat + (N,):
        raise ValueError(f'torchrua_b200: selective_scan A must be (*feat, N) = {feat + (N,)}, got {tuple(A.shape)}')
    if initial is not None and tuple(initial.shape) != (B,) + feat + (N,):
        raise ValueError(f'torchrua_b200: selective_scan initial must be (batch, *feat, N) = {(B,) + feat + (N,)}, '
                         f'got {tuple(initial.shape)}')
    require_cuda(data, delta, A, Bm, Cm, initial)
    return feat, N


def _ssm_forward_raw(x: Tensor, dl: Tensor, A: Tensor, Bm: Tensor, Cm: Tensor, h0: Optional[Tensor], rg: Ragged,
                     side: SideSpec, reverse: bool, want_final: bool, keep_state: bool):
    """(y, final or None, state or None); x, dl (side.rows, H), A (H, N), Bm, Cm (side.rows, N), h0 (B, H, N) or None,
    all contiguous."""
    lib = _lib.load()
    H, N = A.shape
    dt = _DTYPES[x.dtype]
    y = torch.empty_like(x)
    fin = torch.empty((rg.B, H, N), dtype=A.dtype, device=x.device) if want_final else None
    state = None
    if keep_state:
        state = torch.empty(lib.rua_ssm_state_bytes(side.rows, rg.B, H, N, dt), dtype=torch.uint8, device=x.device)
    c_rg, c_side = rg.c_struct(), side.c_struct()
    with _on(x.device):
        prof = _profile_begin()
        _lib.check(lib.rua_ssm_forward(x.data_ptr(), dl.data_ptr(), A.data_ptr(), Bm.data_ptr(), Cm.data_ptr(), _ptr(h0),
                                       y.data_ptr(), _ptr(fin), _ptr(state) if state is not None and state.numel() else None,
                                       H, N, dt, int(reverse), ctypes.byref(c_rg), ctypes.byref(c_side), None, 0,
                                       _stream()), 'rua_ssm_forward')
        if prof is not None:
            # x and delta read once, y written once, B and C read once per channel block + checkpoints
            nb = 3 * x.numel() * x.element_size() + 2 * Bm.numel() * Bm.element_size() + \
                (state.numel() if state is not None else 0)
            _profile_end(prof, 'ssm_forward', nb + 8 * rg.B + (8 * (rg.Tp + rg.B) if side.layout == PACK else 0))
    return y, fin, state


def _ssm_backward_raw(g: Tensor, x: Tensor, dl: Tensor, A: Tensor, Bm: Tensor, Cm: Tensor, state: Tensor, rg: Ragged,
                      side: SideSpec, reverse: bool, want):
    """(grad_x, grad_delta, grad_A, grad_B, grad_C, grad_initial), None where ``want`` is False; inputs contiguous."""
    lib = _lib.load()
    H, N = A.shape
    dt = _DTYPES[x.dtype]
    outs = (torch.empty_like(x) if want[0] else None, torch.empty_like(x) if want[1] else None,
            torch.empty_like(A) if want[2] else None, torch.empty_like(Bm) if want[3] else None,
            torch.empty_like(Cm) if want[4] else None,
            torch.empty((rg.B, H, N), dtype=A.dtype, device=x.device) if want[5] else None)
    if not any(want):
        return outs
    c_rg, c_side = rg.c_struct(), side.c_struct()
    with _on(x.device):
        nbytes = lib.rua_ssm_workspace_bytes(side.rows, rg.B, H, N, dt) if any(want[2:5]) else 0
        ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
        prof = _profile_begin()
        _lib.check(lib.rua_ssm_backward(g.data_ptr(), x.data_ptr(), dl.data_ptr(), A.data_ptr(), Bm.data_ptr(),
                                        Cm.data_ptr(), _ptr(state) if state.numel() else None, *(_ptr(t) for t in outs),
                                        H, N, dt, int(reverse), ctypes.byref(c_rg), ctypes.byref(c_side),
                                        ws.data_ptr() if nbytes else None, nbytes, _stream()), 'rua_ssm_backward')
        if prof is not None:
            # grad_out, x and delta read twice (recompute + adjoint), grad_x and grad_delta written once + checkpoints
            e = x.element_size()
            nb = x.numel() * e * (6 + want[0] + want[1]) + state.numel() + 2 * nbytes
            _profile_end(prof, 'ssm_backward', nb + 8 * rg.B + (8 * (rg.Tp + rg.B) if side.layout == PACK else 0))
    return outs


class _SelectiveScan(torch.autograd.Function):
    """(y, final or None); final is not differentiable.  Once-differentiable: the backward is a native kernel, double
    backward is not supported."""

    @staticmethod
    def forward(ctx, x: Tensor, dl: Tensor, A: Tensor, Bm: Tensor, Cm: Tensor, h0: Optional[Tensor], rg: Ragged,
                side: SideSpec, reverse: bool, want_final: bool):
        xs, ds, As, Bs, Cs = (t.detach().contiguous() for t in (x, dl, A, Bm, Cm))
        hs = None if h0 is None else h0.detach().contiguous()
        y, fin, state = _ssm_forward_raw(xs, ds, As, Bs, Cs, hs, rg, side, reverse, want_final, True)
        if fin is not None:
            ctx.mark_non_differentiable(fin)
        ctx.meta = (rg, side, reverse, h0 is not None)
        ctx.save_for_backward(xs, ds, As, Bs, Cs, state)
        return y, fin

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_y: Optional[Tensor], grad_fin: Optional[Tensor]):
        rg, side, reverse, has_h0 = ctx.meta
        x, dl, A, Bm, Cm, state = ctx.saved_tensors
        need = ctx.needs_input_grad
        want = (need[0], need[1], need[2], need[3], need[4], need[5] and has_h0)
        g = grad_y.contiguous() if grad_y is not None else torch.zeros_like(x)
        return (*_ssm_backward_raw(g, x, dl, A, Bm, Cm, state, rg, side, reverse, want), None, None, None, None)


def selective_scan(data: Tensor, delta: Tensor, A: Tensor, Bm: Tensor, Cm: Tensor, initial: Optional[Tensor],
                   rg: Ragged, side: SideSpec, reverse: bool, want_final: bool) -> Tuple[Tensor, Optional[Tensor]]:
    """(y like data, final (B, *feat, N) or None) of the selective scan over the flattened storage: data, delta
    (side.rows, *feat), Bm, Cm (side.rows, N), A (*feat, N), initial (B, *feat, N) or None; checked by the caller
    (ssm_check); ``rg`` has its pack side."""
    rows, feat, N = data.shape[0], tuple(data.shape[1:]), A.shape[-1]
    H = int(np.prod(feat))
    args = (data.reshape(rows, H), delta.reshape(rows, H), A.reshape(H, N), Bm, Cm,
            None if initial is None else initial.reshape(rg.B, H, N))
    grad = torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in (data, delta, A, Bm, Cm, initial))
    if grad:
        y, fin = _SelectiveScan.apply(*args, rg, side, reverse, want_final)
    else:
        y, fin, _ = _ssm_forward_raw(*(None if t is None else t.contiguous() for t in args), rg, side, reverse,
                                     want_final, False)
    return y.view(data.shape), None if fin is None else fin.view((rg.B,) + feat + (N,))


# ------------------------------------------------------------------------------------------------
# K11: per-sequence Mamba-2 (SSD) state-space scan (+ autograd)
# ------------------------------------------------------------------------------------------------
SSD_MAX_P = 64
SSD_MAX_N = 128


def ssd_check(data: Tensor, delta: Tensor, A: Tensor, Bm: Tensor, Cm: Tensor, initial: Optional[Tensor], B: int,
              lead: int) -> Tuple[int, int, int, int]:
    """validate an SSD scan over ``data`` (*rows, H, P) with ``lead`` row dimensions -> (H, P, G, N), before any device
    work."""
    if data.dtype not in _DTYPES:
        raise RuntimeError(f'torchrua_b200: ssd supports float16/bfloat16/float32/float64, got {data.dtype}')
    acc = _crf_acc_dtype(data.dtype)
    for name, t, want in (('delta', delta, data.dtype), ('B', Bm, data.dtype), ('C', Cm, data.dtype), ('A', A, acc),
                          ('initial', initial, acc)):
        if t is not None and t.dtype != want:
            raise RuntimeError(f'torchrua_b200: ssd {name} must have dtype {want} for a {data.dtype} input, '
                               f'got {t.dtype}')
    if data.dim() != lead + 2:
        raise ValueError(f'torchrua_b200: ssd input must be {lead} row dimension(s) + (H, P), '
                         f'got shape {tuple(data.shape)}')
    rows, (H, P) = tuple(data.shape[:lead]), tuple(data.shape[lead:])
    if tuple(delta.shape) != rows + (H,):
        raise ValueError(f'torchrua_b200: ssd delta must be {rows + (H,)}, got {tuple(delta.shape)}')
    if Bm.dim() != lead + 2 or tuple(Bm.shape[:lead]) != rows:
        raise ValueError(f'torchrua_b200: ssd B must be {rows} + (G, N), got {tuple(Bm.shape)}')
    G, N = Bm.shape[lead:]
    if tuple(Cm.shape) != tuple(Bm.shape):
        raise ValueError(f'torchrua_b200: ssd C must have the shape of B {tuple(Bm.shape)}, got {tuple(Cm.shape)}')
    if G < 1 or H % G:
        raise ValueError(f'torchrua_b200: ssd needs the heads H = {H} to split into G = {G} groups')
    if not 1 <= P <= SSD_MAX_P:
        raise ValueError(f'torchrua_b200: ssd supports head dims 1..{SSD_MAX_P}, got {P}')
    if not 1 <= N <= SSD_MAX_N:
        raise ValueError(f'torchrua_b200: ssd supports state sizes 1..{SSD_MAX_N}, got {N}')
    if tuple(A.shape) != (H,):
        raise ValueError(f'torchrua_b200: ssd A must be (H,) = {(H,)}, got {tuple(A.shape)}')
    if initial is not None and tuple(initial.shape) != (B, H, P, N):
        raise ValueError(f'torchrua_b200: ssd initial must be (batch, H, P, N) = {(B, H, P, N)}, '
                         f'got {tuple(initial.shape)}')
    require_cuda(data, delta, A, Bm, Cm, initial)
    return H, P, G, N


def _ssd_forward_raw(x: Tensor, dl: Tensor, A: Tensor, Bm: Tensor, Cm: Tensor, h0: Optional[Tensor], rg: Ragged,
                     side: SideSpec, reverse: bool, want_final: bool):
    """(y, final or None); x (side.rows, H, P), dl (side.rows, H), A (H,), Bm, Cm (side.rows, G, N), h0 (B, H, P, N) or
    None, all contiguous."""
    lib = _lib.load()
    H, P = x.shape[1:]
    G, N = Bm.shape[1:]
    y = torch.empty_like(x)
    fin = torch.empty((rg.B, H, P, N), dtype=A.dtype, device=x.device) if want_final else None
    c_rg, c_side = rg.c_struct(), side.c_struct()
    with _on(x.device):
        prof = _profile_begin()
        _lib.check(lib.rua_ssd_forward(x.data_ptr(), dl.data_ptr(), A.data_ptr(), Bm.data_ptr(), Cm.data_ptr(), _ptr(h0),
                                       y.data_ptr(), _ptr(fin), H, P, G, N, _DTYPES[x.dtype], int(reverse),
                                       ctypes.byref(c_rg), ctypes.byref(c_side), None, 0, _stream()), 'rua_ssd_forward')
        if prof is not None:
            # x and y once, delta once, B and C once per head
            nb = 2 * x.numel() * x.element_size() + dl.numel() * dl.element_size() + \
                2 * Bm.numel() * Bm.element_size() * (H // G)
            _profile_end(prof, 'ssd_forward', nb + 8 * rg.B + (8 * (rg.Tp + rg.B) if side.layout == PACK else 0))
    return y, fin


def _ssd_backward_raw(g: Tensor, x: Tensor, dl: Tensor, A: Tensor, Bm: Tensor, Cm: Tensor, h0: Optional[Tensor],
                      rg: Ragged, side: SideSpec, reverse: bool, want):
    """(grad_x, grad_delta, grad_A, grad_B, grad_C, grad_initial), None where ``want`` is False; inputs contiguous."""
    lib = _lib.load()
    H, P = x.shape[1:]
    G, N = Bm.shape[1:]
    dt = _DTYPES[x.dtype]
    outs = (torch.empty_like(x) if want[0] else None, torch.empty_like(dl) if want[1] else None,
            torch.empty_like(A) if want[2] else None, torch.empty_like(Bm) if want[3] else None,
            torch.empty_like(Cm) if want[4] else None,
            torch.empty((rg.B, H, P, N), dtype=A.dtype, device=x.device) if want[5] else None)
    if not any(want):
        return outs
    c_rg, c_side = rg.c_struct(), side.c_struct()
    with _on(x.device):
        nbytes = lib.rua_ssd_workspace_bytes(side.rows, rg.B, rg.Tp, H, P, G, N, dt)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
        prof = _profile_begin()
        _lib.check(lib.rua_ssd_backward(g.data_ptr(), x.data_ptr(), dl.data_ptr(), A.data_ptr(), Bm.data_ptr(),
                                        Cm.data_ptr(), _ptr(h0), *(_ptr(t) for t in outs), H, P, G, N, dt,
                                        int(reverse), ctypes.byref(c_rg), ctypes.byref(c_side),
                                        ws.data_ptr() if nbytes else None, nbytes, _stream()), 'rua_ssd_backward')
        if prof is not None:
            # x, delta, grad_out twice (recompute + reverse sweep), B and C twice per head, the gradients once
            e = x.element_size()
            nb = x.numel() * e * (3 + want[0]) + dl.numel() * e * (2 + want[1]) + \
                Bm.numel() * e * (4 * (H // G) + want[3] + want[4])
            _profile_end(prof, 'ssd_backward', nb + 8 * rg.B + (8 * (rg.Tp + rg.B) if side.layout == PACK else 0))
    return outs


class _SSD(torch.autograd.Function):
    """(y, final or None); final is not differentiable.  Saves only its inputs: the backward recomputes the states.
    Once-differentiable: the backward is a native kernel, double backward is not supported."""

    @staticmethod
    def forward(ctx, x: Tensor, dl: Tensor, A: Tensor, Bm: Tensor, Cm: Tensor, h0: Optional[Tensor], rg: Ragged,
                side: SideSpec, reverse: bool, want_final: bool):
        xs, ds, As, Bs, Cs = (t.detach().contiguous() for t in (x, dl, A, Bm, Cm))
        hs = None if h0 is None else h0.detach().contiguous()
        y, fin = _ssd_forward_raw(xs, ds, As, Bs, Cs, hs, rg, side, reverse, want_final)
        if fin is not None:
            ctx.mark_non_differentiable(fin)
        ctx.meta = (rg, side, reverse, h0 is not None)
        ctx.save_for_backward(xs, ds, As, Bs, Cs, hs)
        return y, fin

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_y: Optional[Tensor], grad_fin: Optional[Tensor]):
        rg, side, reverse, has_h0 = ctx.meta
        x, dl, A, Bm, Cm, h0 = ctx.saved_tensors
        need = ctx.needs_input_grad
        want = (need[0], need[1], need[2], need[3], need[4], need[5] and has_h0)
        g = grad_y.contiguous() if grad_y is not None else torch.zeros_like(x)
        return (*_ssd_backward_raw(g, x, dl, A, Bm, Cm, h0, rg, side, reverse, want), None, None, None, None)


def ssd(data: Tensor, delta: Tensor, A: Tensor, Bm: Tensor, Cm: Tensor, initial: Optional[Tensor], rg: Ragged,
        side: SideSpec, reverse: bool, want_final: bool) -> Tuple[Tensor, Optional[Tensor]]:
    """(y like data, final (B, H, P, N) or None) of the SSD scan over the flattened storage: data (side.rows, H, P),
    delta (side.rows, H), Bm, Cm (side.rows, G, N), A (H,), initial (B, H, P, N) or None; checked by the caller
    (ssd_check); ``rg`` has its pack side."""
    args = (data, delta, A, Bm, Cm, initial)
    grad = torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in args)
    if grad:
        return _SSD.apply(*args, rg, side, reverse, want_final)
    return _ssd_forward_raw(*(None if t is None else t.contiguous() for t in args), rg, side, reverse, want_final)


# ------------------------------------------------------------------------------------------------
# K12: per-sequence gated delta rule (Gated DeltaNet) (+ autograd)
# ------------------------------------------------------------------------------------------------
GDN_MAX_K = 128
GDN_MAX_V = 256


def gdn_check(data: Tensor, q: Tensor, k: Tensor, g: Tensor, beta: Tensor, initial: Optional[Tensor], B: int,
              lead: int) -> Tuple[int, int, int, int]:
    """validate a gated delta rule over ``data`` (*rows, H, V) with ``lead`` row dimensions -> (H, G, K, V), before any
    device work."""
    if data.dtype not in _DTYPES:
        raise RuntimeError(f'torchrua_b200: gated_delta_rule supports float16/bfloat16/float32/float64, got {data.dtype}')
    acc = _crf_acc_dtype(data.dtype)
    for name, t, want in (('q', q, data.dtype), ('k', k, data.dtype), ('beta', beta, data.dtype), ('g', g, acc),
                          ('initial', initial, acc)):
        if t is not None and t.dtype != want:
            raise RuntimeError(f'torchrua_b200: gated_delta_rule {name} must have dtype {want} for a {data.dtype} '
                               f'input, got {t.dtype}')
    if data.dim() != lead + 2:
        raise ValueError(f'torchrua_b200: gated_delta_rule input must be {lead} row dimension(s) + (H, V), '
                         f'got shape {tuple(data.shape)}')
    rows, (H, V) = tuple(data.shape[:lead]), tuple(data.shape[lead:])
    if q.dim() != lead + 2 or tuple(q.shape[:lead]) != rows:
        raise ValueError(f'torchrua_b200: gated_delta_rule q must be {rows} + (G, K), got {tuple(q.shape)}')
    G, K = q.shape[lead:]
    if tuple(k.shape) != tuple(q.shape):
        raise ValueError(f'torchrua_b200: gated_delta_rule k must have the shape of q {tuple(q.shape)}, '
                         f'got {tuple(k.shape)}')
    for name, t in (('g', g), ('beta', beta)):
        if tuple(t.shape) != rows + (H,):
            raise ValueError(f'torchrua_b200: gated_delta_rule {name} must be {rows + (H,)}, got {tuple(t.shape)}')
    if G < 1 or H % G:
        raise ValueError(f'torchrua_b200: gated_delta_rule needs the value heads H = {H} to split into G = {G} groups')
    if not 1 <= K <= GDN_MAX_K:
        raise ValueError(f'torchrua_b200: gated_delta_rule supports key dims 1..{GDN_MAX_K}, got {K}')
    if not 1 <= V <= GDN_MAX_V:
        raise ValueError(f'torchrua_b200: gated_delta_rule supports value dims 1..{GDN_MAX_V}, got {V}')
    if initial is not None and tuple(initial.shape) != (B, H, K, V):
        raise ValueError(f'torchrua_b200: gated_delta_rule initial must be (batch, H, K, V) = {(B, H, K, V)}, '
                         f'got {tuple(initial.shape)}')
    require_cuda(data, q, k, g, beta, initial)
    return H, G, K, V


def gdn_scale(scale: Optional[float], K: int) -> float:
    """the output scale: K^-1/2 when None"""
    return float(K) ** -0.5 if scale is None else float(scale)


def _gdn_forward_raw(v: Tensor, q: Tensor, k: Tensor, g: Tensor, beta: Tensor, h0: Optional[Tensor], scale: float,
                     rg: Ragged, side: SideSpec, reverse: bool, want_final: bool):
    """(o, final or None); v (side.rows, H, V), q, k (side.rows, G, K), g, beta (side.rows, H), h0 (B, H, K, V) or None,
    all contiguous."""
    lib = _lib.load()
    H, V = v.shape[1:]
    G, K = q.shape[1:]
    o = torch.empty_like(v)
    fin = torch.empty((rg.B, H, K, V), dtype=g.dtype, device=v.device) if want_final else None
    c_rg, c_side = rg.c_struct(), side.c_struct()
    with _on(v.device):
        prof = _profile_begin()
        _lib.check(lib.rua_gdn_forward(v.data_ptr(), q.data_ptr(), k.data_ptr(), g.data_ptr(), beta.data_ptr(), _ptr(h0),
                                       o.data_ptr(), _ptr(fin), H, G, K, V, scale, _DTYPES[v.dtype], int(reverse),
                                       ctypes.byref(c_rg), ctypes.byref(c_side), None, 0, _stream()), 'rua_gdn_forward')
        if prof is not None:
            # v and o once, g and beta once, q and k once per value head block
            nb = 2 * v.numel() * v.element_size() + g.numel() * g.element_size() + beta.numel() * beta.element_size() + \
                2 * q.numel() * q.element_size() * (H // G) * ((V + 63) // 64)
            _profile_end(prof, 'gdn_forward', nb + 8 * rg.B + (8 * (rg.Tp + rg.B) if side.layout == PACK else 0))
    return o, fin


def _gdn_backward_raw(go: Tensor, v: Tensor, q: Tensor, k: Tensor, g: Tensor, beta: Tensor, h0: Optional[Tensor],
                      scale: float, rg: Ragged, side: SideSpec, reverse: bool, want):
    """(grad_v, grad_q, grad_k, grad_g, grad_beta, grad_initial), None where ``want`` is False; inputs contiguous."""
    lib = _lib.load()
    H, V = v.shape[1:]
    G, K = q.shape[1:]
    dt = _DTYPES[v.dtype]
    outs = (torch.empty_like(v) if want[0] else None, torch.empty_like(q) if want[1] else None,
            torch.empty_like(k) if want[2] else None, torch.empty_like(g) if want[3] else None,
            torch.empty_like(beta) if want[4] else None,
            torch.empty((rg.B, H, K, V), dtype=g.dtype, device=v.device) if want[5] else None)
    if not any(want):
        return outs
    c_rg, c_side = rg.c_struct(), side.c_struct()
    with _on(v.device):
        nbytes = lib.rua_gdn_workspace_bytes(side.rows, rg.B, rg.Tp, H, G, K, V, dt)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=v.device)
        prof = _profile_begin()
        _lib.check(lib.rua_gdn_backward(go.data_ptr(), v.data_ptr(), q.data_ptr(), k.data_ptr(), g.data_ptr(),
                                        beta.data_ptr(), _ptr(h0), *(_ptr(t) for t in outs), H, G, K, V, scale, dt,
                                        int(reverse), ctypes.byref(c_rg), ctypes.byref(c_side),
                                        ws.data_ptr() if nbytes else None, nbytes, _stream()), 'rua_gdn_backward')
        if prof is not None:
            # v and grad_out twice (recompute + reverse sweep), q and k three times per head block, the gradients once
            e = v.element_size()
            nb = v.numel() * e * (4 + want[0]) + q.numel() * e * (6 * (H // G) * ((V + 63) // 64) + want[1] + want[2])
            _profile_end(prof, 'gdn_backward', nb + 8 * rg.B + (8 * (rg.Tp + rg.B) if side.layout == PACK else 0))
    return outs


class _GDN(torch.autograd.Function):
    """(o, final or None); final is not differentiable.  Saves only its inputs: the backward recomputes the states.
    Once-differentiable: the backward is a native kernel, double backward is not supported."""

    @staticmethod
    def forward(ctx, v: Tensor, q: Tensor, k: Tensor, g: Tensor, beta: Tensor, h0: Optional[Tensor], scale: float,
                rg: Ragged, side: SideSpec, reverse: bool, want_final: bool):
        vs, qs, ks, gs, bs = (t.detach().contiguous() for t in (v, q, k, g, beta))
        hs = None if h0 is None else h0.detach().contiguous()
        o, fin = _gdn_forward_raw(vs, qs, ks, gs, bs, hs, scale, rg, side, reverse, want_final)
        if fin is not None:
            ctx.mark_non_differentiable(fin)
        ctx.meta = (scale, rg, side, reverse, h0 is not None)
        ctx.save_for_backward(vs, qs, ks, gs, bs, hs)
        return o, fin

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_o: Optional[Tensor], grad_fin: Optional[Tensor]):
        scale, rg, side, reverse, has_h0 = ctx.meta
        v, q, k, g, beta, h0 = ctx.saved_tensors
        need = ctx.needs_input_grad
        want = (need[0], need[1], need[2], need[3], need[4], need[5] and has_h0)
        go = grad_o.contiguous() if grad_o is not None else torch.zeros_like(v)
        return (*_gdn_backward_raw(go, v, q, k, g, beta, h0, scale, rg, side, reverse, want),
                None, None, None, None, None)


def gdn(data: Tensor, q: Tensor, k: Tensor, g: Tensor, beta: Tensor, initial: Optional[Tensor], scale: float,
        rg: Ragged, side: SideSpec, reverse: bool, want_final: bool) -> Tuple[Tensor, Optional[Tensor]]:
    """(o like data, final (B, H, K, V) or None) of the gated delta rule over the flattened storage: data (side.rows, H,
    V), q, k (side.rows, G, K), g, beta (side.rows, H), initial (B, H, K, V) or None; checked by the caller (gdn_check);
    ``rg`` has its pack side."""
    args = (data, q, k, g, beta, initial)
    grad = torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in args)
    if grad:
        return _GDN.apply(*args, scale, rg, side, reverse, want_final)
    return _gdn_forward_raw(*(None if t is None else t.contiguous() for t in args), scale, rg, side, reverse, want_final)


# ------------------------------------------------------------------------------------------------
# scatter_*: stable sort of the index + bucket boundaries + segment reduce over GATHERED rows
# ------------------------------------------------------------------------------------------------
def sort_keys(keys: Tensor, max_key: int) -> Tuple[Tensor, Tensor]:
    """stable ascending argsort of int64 keys in [0, max_key] (device radix sort) and its inverse."""
    lib = _lib.load()
    keys = _i64(keys)
    require_cuda(keys)
    n = keys.numel()
    srt = torch.empty(n, dtype=torch.long, device=keys.device)
    uns = torch.empty(n, dtype=torch.long, device=keys.device)
    if n > 0:
        with _on(keys.device):
            nbytes = lib.rua_sort_workspace_bytes(n)
            ws = torch.empty(nbytes, dtype=torch.uint8, device=keys.device)
            _lib.check(lib.rua_sort_keys(keys.data_ptr(), n, max(max_key, 0), srt.data_ptr(), uns.data_ptr(),
                                         ws.data_ptr(), nbytes, _stream()), 'rua_sort_keys')
    return srt, uns


def bucket_offsets(keys: Tensor, srt: Tensor, buckets: int) -> Tensor:
    """off[m] = #{k : keys[k] < m} for m in [0, buckets], given the ascending permutation of the keys."""
    lib = _lib.load()
    keys = _i64(keys)
    off = torch.empty(buckets + 1, dtype=torch.long, device=keys.device)
    with _on(keys.device):
        _lib.check(lib.rua_bucket_offsets(_ptr(keys), _ptr(srt), keys.numel(), buckets, off.data_ptr(), _stream()),
                   'rua_bucket_offsets')
    return off


class _ScatterReduce(torch.autograd.Function):
    """out[m] = reduce over {source[k] : index[k] == m}; rows of `source` are gathered in sorted-index order
    inside the kernel.  Backward: gather the rows into sorted order, run the segment-reduce backward kernel,
    scatter the gradient rows back -- every row is touched by exactly one thread, no atomics."""

    @staticmethod
    def forward(ctx, source: Tensor, srt: Tensor, off: Tensor, S: int, op: int):
        flat = source.detach()
        if not flat.is_contiguous():
            flat = flat.contiguous()
        out = _reduce_raw(flat, off, S, op, rows=srt)
        ctx.op, ctx.S = op, S
        ctx.save_for_backward(flat, srt, off, out)
        return out

    @staticmethod
    def backward(ctx, grad_out: Tensor):
        source, srt, off, out = ctx.saved_tensors
        K = srt.numel()
        H = source[0].numel() if source.shape[0] else 0
        grad = torch.zeros_like(source)
        if K > 0 and H > 0:
            ordered = _gather_rows_raw(source, srt)               # rows in sorted-index order
            grad_ordered = torch.empty_like(ordered)
            _reduce_backward_raw(grad_out.contiguous(), out, ordered, off, ctx.S, ctx.op, grad_ordered)
            scatter_rows_(grad, srt, grad_ordered)
        return grad, None, None, None, None


def segment_reduce_gathered(source: Tensor, rows: Tensor, segment_sizes: Tensor, op: str) -> Tensor:
    """segment_reduce(source[rows], segment_sizes, op) without materialising ``source[rows]``: the kernel reads row
    ``rows[j]`` where the plain reduction reads row ``j``.  ``rows`` must not repeat (backward scatters the gradient rows)."""
    require_cuda(source, rows, segment_sizes)
    rg = ragged_from_lengths(segment_sizes)
    rows = _i64(rows).view(-1)
    if source.requires_grad and torch.is_grad_enabled():
        return _ScatterReduce.apply(source, rows, rg.off, rg.B, _OPS[op])
    return _reduce_raw(source if source.is_contiguous() else source.contiguous(), rg.off, rg.B, _OPS[op], rows=rows)


def scatter_reduce(source: Tensor, index: Tensor, buckets: int, op: str):
    """(reduced (buckets, *feat), counts (buckets,)) of `source` rows grouped by `index` along dim 0."""
    require_cuda(source, index)
    srt, _ = sort_keys(index, buckets - 1)
    off = bucket_offsets(index, srt, buckets)
    if source.requires_grad and torch.is_grad_enabled():
        red = _ScatterReduce.apply(source, srt, off, buckets, _OPS[op])
    else:
        red = _reduce_raw(source if source.is_contiguous() else source.contiguous(), off, buckets, _OPS[op], rows=srt)
    return red, off[1:] - off[:-1]
