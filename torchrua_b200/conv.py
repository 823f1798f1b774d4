"""Per-sequence depthwise 1-D convolution along the time axis of every sequence, never crossing from one sequence into
the next.  The reference has no counterpart; without it a user pads (``x.left(0)``), runs ``F.conv1d(groups=H)`` on the
transposed ``(B, H, T)`` batch and unpads -- which moves the padding twice -- or runs ``F.conv1d`` straight on the
storage, which mixes every sequence's first and last ``K - 1`` outputs with its neighbours.

For token ``(i, t)`` of sequence ``i`` (length ``len_i``), feature column ``h``, kernel size ``K`` and left padding ``p``::

    y(i, t, h) = bias[h] + sum_{k<K} weight[h, k] * x(i, t + k - p, h),   x(i, s, .) = 0 for s outside [0, len_i)

``padding='causal'`` is ``p = K - 1`` (``weight[..., K-1]`` multiplies the current token, as in ``causal_conv1d``),
``padding='same'`` is ``p = (K - 1) // 2`` (torch's ``padding='same'``), an int is ``p`` itself (``0 <= p <= K - 1``).
There is no default: neither convention should be silent.  ``1 <= K <= 32``.

One native kernel (rua_segment_conv) serves every layout: it reads the rows where they lie (C, L, P or R storage), so the
result keeps the layout and the metadata of its input.  Rows that hold no token (L / R padding, C rows past
``sum(segment_sizes)``) are copied through, and their gradient passes through.  ``weight`` and ``bias`` have the
payload's dtype, as ``F.conv1d`` requires.  Accumulation is fp32 (fp64 for fp64) with one rounding;
``strict_reductions()`` does not apply.  Gradients reach the input, the weight and the bias (the weight and bias
gradients are bit-identical run to run); the backward is once-differentiable, double backward raises.
"""
from typing import Optional

from torch import Tensor

from torchrua_b200 import _native
from torchrua_b200._lib import CAT, LEFT, PACK, RIGHT
from torchrua_b200._native import SideSpec
from torchrua_b200.layout import C, L, P, R

__all__ = ['segment_depthwise_conv1d']


def segment_depthwise_conv1d(tensor: Tensor, segment_sizes: Tensor, weight: Tensor, bias: Optional[Tensor] = None, *,
                             padding) -> Tensor:
    """depthwise convolution of every segment of ``tensor`` (N, *feat) in C order; ``segment_sizes`` (S,) int64,
    ``weight`` (*feat, K), ``bias`` (*feat) or None, ``padding`` 'causal', 'same' or an int."""
    _native.conv_check(tensor, weight, bias, tuple(tensor.shape[1:]), padding)
    _native.require_cuda(segment_sizes)
    rg = _native.ragged_from_lengths(segment_sizes)
    return _native.segment_conv(tensor, weight, bias, padding, rg, SideSpec(CAT, rows=tensor.size()[0]))


# ---------------------------------------------------------------------------------------------------------------------
# methods on the four layouts: the convolution runs on the flattened storage, the result keeps the metadata
# ---------------------------------------------------------------------------------------------------------------------
def _flat_conv(self, weight: Tensor, bias: Optional[Tensor] = None, *, padding):
    """C / P: ``data`` is (N, *feat)."""
    _native.conv_check(self.data, weight, bias, tuple(self.data.shape[1:]), padding)
    rg = self._ragged()
    side = SideSpec(CAT if isinstance(self, C) else PACK, rows=self.data.size()[0])
    return self._replace(data=_native.segment_conv(self.data, weight, bias, padding, rg, side))


def _padded_conv(self, weight: Tensor, bias: Optional[Tensor] = None, *, padding):
    """L / R: ``data`` is (B, W, *feat)."""
    _native.conv_check(self.data, weight, bias, tuple(self.data.shape[2:]), padding)
    rg = self._ragged()
    b, w = self.data.size()[:2]
    side = SideSpec(RIGHT if self._right_aligned else LEFT, width=w, rows=b * w)
    out = _native.segment_conv(self.data.flatten(start_dim=0, end_dim=1), weight, bias, padding, rg, side)
    return self._replace(data=out.view(self.data.size()))


def _bind(cls, run):
    def depthwise_conv1d(self, weight: Tensor, bias: Optional[Tensor] = None, *, padding):
        """per-sequence depthwise 1-D convolution along time (see ``torchrua_b200.conv``); same layout and metadata."""
        return run(self, weight, bias, padding=padding)

    cls.depthwise_conv1d = depthwise_conv1d


_bind(C, _flat_conv)
_bind(P, _flat_conv)
_bind(L, _padded_conv)
_bind(R, _padded_conv)
