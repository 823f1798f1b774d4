"""Per-sequence prefix scans: cumsum, logcumsumexp, cummax and cummin along the time axis of every sequence, restarting
at every sequence boundary.  The reference has no counterpart; without these a user pads (``x.left(fill)``), runs the
torch scan along dim 1 and unpads, which moves the padding twice and needs a per-op fill.

One native kernel (rua_segment_scan) serves every layout: it reads the rows where they lie (C, L, P or R storage), so
the result keeps the layout and the metadata of its input.  ``reverse=True`` scans every sequence from its end, like
``x.rev()`` -> scan -> ``.rev()``; the indices of cummax / cummin are positions within the sequence either way.  Rows
that hold no token (L / R padding, C rows past ``sum(segment_sizes)``) are copied through, with index 0.

Accumulation is fp32 (fp64 for fp64) with one rounding; ``strict_reductions()`` does not apply to scans.

``segment_linear_recurrence`` / ``.linear_recurrence`` run the diagonal gated linear recurrence of Mamba-, minGRU-,
Griffin- and GLA-style blocks on the same kernel, per token ``(i, t)`` and feature column::

    reverse=False:  h(i, t) = gate(i, t) * h(i, t - 1) + x(i, t),   h(i, -1)    = initial[i] (0 without one)
    reverse=True:   h(i, t) = gate(i, t) * h(i, t + 1) + x(i, t),   h(i, len_i) = initial[i]

``gate`` has the shape, dtype and layout of the payload and may take any real value (0 resets the state, 1 gives
cumsum).  ``initial`` is ``(B, *feat)`` in ``token_sizes`` order (for P the original sequence index).  To continue a
recurrence over the next chunk of every sequence, pass ``y.last()`` (``y.head()`` for reverse) as its ``initial``.
Results are deterministic run to run.  Behaviour is specified for finite inputs: non-finite values propagate, but the
combination order differs from a sequential loop, so where they appear (``0 * inf``, for one) may differ.  Rows that
hold no token are copied through; their ``x`` gradient passes ``grad_out`` through and their gate gradient is 0.
Gradients reach ``x``, ``gate`` and ``initial`` (0 for an empty sequence); double backward raises.
"""
from typing import Optional, Tuple

import torch
from torch import Tensor

from torchrua_b200 import _native
from torchrua_b200._lib import CAT, LEFT, PACK, RIGHT
from torchrua_b200._native import SideSpec
from torchrua_b200.layout import C, L, P, R

__all__ = ['segment_cumsum', 'segment_logcumsumexp', 'segment_cummax', 'segment_cummin', 'segment_linear_recurrence']


def _segment_scan(tensor: Tensor, segment_sizes: Tensor, op: str, reverse: bool):
    _native._scan_check(tensor)
    _native.require_cuda(tensor, segment_sizes)
    rg = _native.ragged_from_lengths(segment_sizes)
    return _native.segment_scan(tensor, rg, SideSpec(CAT, rows=tensor.size()[0]), op, reverse)


def segment_cumsum(tensor: Tensor, segment_sizes: Tensor, reverse: bool = False) -> Tensor:
    """running sum of every segment of ``tensor`` (N, *) in C order; ``segment_sizes`` (S,) int64."""
    return _segment_scan(tensor, segment_sizes, 'sum', reverse)[0]


def segment_logcumsumexp(tensor: Tensor, segment_sizes: Tensor, reverse: bool = False) -> Tensor:
    """running log-sum-exp of every segment.  Its gradient is 0 where the input is -inf (torch gives NaN for a leading
    -inf)."""
    return _segment_scan(tensor, segment_sizes, 'logsumexp', reverse)[0]


def segment_cummax(tensor: Tensor, segment_sizes: Tensor, reverse: bool = False):
    """(values, indices) of the running maximum of every segment; indices are positions within the segment, ties and
    NaN as torch.cummax."""
    return torch.return_types.cummax(_segment_scan(tensor, segment_sizes, 'max', reverse))


def segment_cummin(tensor: Tensor, segment_sizes: Tensor, reverse: bool = False):
    """(values, indices) of the running minimum of every segment, as segment_cummax."""
    return torch.return_types.cummin(_segment_scan(tensor, segment_sizes, 'min', reverse))


def segment_linear_recurrence(tensor: Tensor, segment_sizes: Tensor, gate: Tensor, initial: Optional[Tensor] = None,
                              reverse: bool = False) -> Tensor:
    """h_t = gate_t * h_(t-1) + x_t along every segment of ``tensor`` (N, *feat) in C order; ``segment_sizes`` (S,)
    int64, ``gate`` (N, *feat), ``initial`` (S, *feat) or None."""
    _native.linrec_check(tensor, gate, initial, segment_sizes.shape[0], tuple(tensor.shape[1:]))
    _native.require_cuda(tensor, segment_sizes)
    rg = _native.ragged_from_lengths(segment_sizes)
    return _native.linear_recurrence(tensor, gate, initial, rg, SideSpec(CAT, rows=tensor.size()[0]), reverse)


# ---------------------------------------------------------------------------------------------------------------------
# methods on the four layouts: the scan runs on the flattened storage, the result is rebuilt with the same metadata
# ---------------------------------------------------------------------------------------------------------------------
def _cat_scan(self: C, op: str, reverse: bool) -> Tuple[Tensor, Tensor]:
    _native._scan_check(self.data)
    rg = self._ragged()
    return _native.segment_scan(self.data, rg, SideSpec(CAT, rows=self.data.size()[0]), op, reverse)


def _padded_scan(self, op: str, reverse: bool) -> Tuple[Tensor, Tensor]:
    _native._scan_check(self.data)
    rg = self._ragged()
    b, w = self.data.size()[:2]
    side = SideSpec(RIGHT if self._right_aligned else LEFT, width=w, rows=b * w)
    out, idx = _native.segment_scan(self.data.flatten(start_dim=0, end_dim=1), rg, side, op, reverse)
    shape = self.data.size()
    return out.view(shape), (None if idx is None else idx.view(shape))


def _pack_scan(self: P, op: str, reverse: bool) -> Tuple[Tensor, Tensor]:
    _native._scan_check(self.data)
    rg = self._ragged()
    return _native.segment_scan(self.data, rg, SideSpec(PACK, rows=self.data.size()[0]), op, reverse)


def _bind(cls, run):
    def cumsum(self, reverse: bool = False):
        return self._replace(data=run(self, 'sum', reverse)[0])

    def logcumsumexp(self, reverse: bool = False):
        return self._replace(data=run(self, 'logsumexp', reverse)[0])

    def cummax(self, reverse: bool = False):
        out, idx = run(self, 'max', reverse)
        return self._replace(data=out), self._replace(data=idx)

    def cummin(self, reverse: bool = False):
        out, idx = run(self, 'min', reverse)
        return self._replace(data=out), self._replace(data=idx)

    for fn in (cumsum, logcumsumexp, cummax, cummin):
        setattr(cls, fn.__name__, fn)


def _flat_linrec(self, gate: Tensor, initial: Optional[Tensor] = None, reverse: bool = False):
    """C / P: ``data`` is (N, *feat)."""
    cat = isinstance(self, C)
    if cat:
        B = self.token_sizes.shape[0]
    elif self.unsorted_indices is not None:
        B = self.unsorted_indices.numel()
    else:
        B = int(self.batch_sizes[0]) if self.batch_sizes.numel() else 0
    _native.linrec_check(self.data, gate, initial, B, tuple(self.data.shape[1:]))
    rg = self._ragged()
    side = SideSpec(CAT if cat else PACK, rows=self.data.size()[0])
    return self._replace(data=_native.linear_recurrence(self.data, gate, initial, rg, side, reverse))


def _padded_linrec(self, gate: Tensor, initial: Optional[Tensor] = None, reverse: bool = False):
    """L / R: ``data`` is (B, W, *feat); the gate at padding positions is ignored."""
    _native.linrec_check(self.data, gate, initial, self.data.shape[0], tuple(self.data.shape[2:]))
    rg = self._ragged()
    b, w = self.data.size()[:2]
    side = SideSpec(RIGHT if self._right_aligned else LEFT, width=w, rows=b * w)
    out = _native.linear_recurrence(self.data.flatten(start_dim=0, end_dim=1), gate.flatten(start_dim=0, end_dim=1),
                                    initial, rg, side, reverse)
    return self._replace(data=out.view(self.data.size()))


def _bind_linrec(cls, run):
    def linear_recurrence(self, gate: Tensor, initial: Optional[Tensor] = None, reverse: bool = False):
        """per-sequence h_t = gate_t * h_(t-1) + x_t along time (see ``torchrua_b200.scan``); same layout and
        metadata."""
        return run(self, gate, initial, reverse)

    cls.linear_recurrence = linear_recurrence


_bind(C, _cat_scan)
_bind(L, _padded_scan)
_bind(R, _padded_scan)
_bind(P, _pack_scan)
_bind_linrec(C, _flat_linrec)
_bind_linrec(P, _flat_linrec)
_bind_linrec(L, _padded_linrec)
_bind_linrec(R, _padded_linrec)
