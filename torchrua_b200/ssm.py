"""Per-sequence selective state-space scan, the recurrence at the core of a Mamba-1 mixer
(in_proj -> causal depthwise conv1d -> SiLU -> x_proj (delta, B, C) -> selective scan -> gate -> out_proj).  The
reference has no counterpart; without it a user pads and loops over ``T`` in Python, keeping a ``(B, H, N)`` state per
step for autograd, or composes it from ``linear_recurrence`` over ``H x N`` columns, which materialises
``(tokens, H, N)`` gates, inputs and states.  Scanning the C storage with a dense-batch implementation instead leaks
state from one sequence into the next.

For token ``(i, t)`` of sequence ``i``, channel ``h`` (the flattened ``*feat``) and state ``n < N``::

    dA_t[h, n] = exp(delta_t[h] * A[h, n])
    h_t[h, n]  = dA_t[h, n] * h_(t-1)[h, n] + delta_t[h] * B_t[n] * x_t[h],    h_(-1) = initial[i] (0 without one)
    y_t[h]     = sum_n C_t[n] * h_t[h, n]
    final[i]   = h at the last token (initial[i], or 0, for an empty sequence)

``reverse=True`` runs from each sequence's end: ``h_t`` depends on ``h_(t+1)``, ``h_(len_i) = initial[i]`` and
``final[i]`` is the state at ``t = 0`` (the convention of ``linear_recurrence``; bidirectional encoders use it).

* ``x`` and ``delta`` have the payload's shape and layout: ``(rows, *feat)``, or ``(B, W, *feat)`` for L and R.  ``B``
  and ``C`` are ``(rows, N)`` in the same layout (``(B, W, N)`` for L and R), shared by every channel.  ``x``,
  ``delta``, ``B`` and ``C`` share one dtype: fp16, bf16, fp32 or fp64.
* ``A`` is ``(*feat, N)``; ``initial`` and ``final`` are ``(batch, *feat, N)`` in ``token_sizes`` order (for P the
  original sequence index).  All three are in the ACCUMULATOR dtype: fp32, or fp64 for fp64 payloads (Mamba's
  ``A = -exp(A_log)`` is an fp32 parameter under bf16, and a carried state in bf16 would lose precision).
* ``1 <= N <= 16``.  Accumulation is fp32 (fp64 for fp64) with one rounding of ``y``, which has the payload dtype.
* Rows that hold no token (L / R padding, C rows past ``sum(sizes)``) are copied through from ``x``; there the ``x``
  gradient passes ``grad_out`` through and the ``delta``, ``B`` and ``C`` gradients are 0.
* Gradients reach ``x``, ``delta``, ``A``, ``B``, ``C`` and ``initial`` (0 for an empty sequence); an unwanted one is not
  computed, and the forward keeps its checkpoints (one state per 32 steps of every sequence) only when a gradient is
  wanted.  ``final`` is not differentiable.  Double backward raises.
* Every result is bit-identical run to run and, for the same sequences, on C, L, P and R: no float atomics, and every
  sum runs in a fixed order.
* Single-token decoding is ``len = 1`` sequences with ``initial``; streaming passes one part's ``final`` as the next
  part's ``initial``.

Out of scope: the fused ``softplus(delta + bias)``, the ``D * x`` skip and the ``silu(z)`` gate (pointwise: write them
in torch), complex ``A``, grouped or per-channel ``B`` / ``C``, ``N > 16``, Mamba-2 / SSD (a scalar decay per head with
a chunked matmul form), and a gradient through ``final``.

One set of native kernels (rua_ssm_forward / rua_ssm_backward) serves every layout, reading the rows where they lie.
"""
from typing import Optional

from torch import Tensor

from torchrua_b200 import _native
from torchrua_b200 import layout
from torchrua_b200._lib import CAT, LEFT, PACK, RIGHT
from torchrua_b200._native import SideSpec

__all__ = ['segment_selective_scan']


def segment_selective_scan(tensor: Tensor, segment_sizes: Tensor, delta: Tensor, A: Tensor, B: Tensor, C: Tensor,
                           initial: Optional[Tensor] = None, reverse: bool = False, return_final_state: bool = False):
    """selective scan along every segment of ``tensor`` (rows, *feat) in C order; ``segment_sizes`` (S,) int64, ``delta``
    like ``tensor``, ``B`` and ``C`` (rows, N), ``A`` (*feat, N), ``initial`` (S, *feat, N) or None -> y, or
    ``(y, final)`` with ``return_final_state``."""
    _native.ssm_check(tensor, delta, A, B, C, initial, segment_sizes.shape[0], 1)
    _native.require_cuda(segment_sizes)
    rg = _native.ragged_from_lengths(segment_sizes, want_pack=True)
    y, fin = _native.selective_scan(tensor, delta, A, B, C, initial, rg, SideSpec(CAT, rows=tensor.size()[0]), reverse,
                                    return_final_state)
    return (y, fin) if return_final_state else y


# ---------------------------------------------------------------------------------------------------------------------
# methods on the four layouts: the scan runs on the flattened storage, the result keeps the layout and the metadata
# ---------------------------------------------------------------------------------------------------------------------
def _batch(self) -> int:
    if isinstance(self, layout.C):
        return self.token_sizes.shape[0]
    if self.unsorted_indices is not None:
        return self.unsorted_indices.numel()
    return int(self.batch_sizes[0]) if self.batch_sizes.numel() else 0


def _flat(self, delta, A, B, C, initial, reverse, want_final):
    """C / P: ``data`` is (rows, *feat)."""
    _native.ssm_check(self.data, delta, A, B, C, initial, _batch(self), 1)
    cat = isinstance(self, layout.C)
    rg = self._ragged(want_pack=True) if cat else self._ragged()
    side = SideSpec(CAT if cat else PACK, rows=self.data.size()[0])
    return _native.selective_scan(self.data, delta, A, B, C, initial, rg, side, reverse, want_final)


def _padded(self, delta, A, B, C, initial, reverse, want_final):
    """L / R: ``data`` is (B, W, *feat); delta, B and C at padding positions are ignored."""
    _native.ssm_check(self.data, delta, A, B, C, initial, self.data.shape[0], 2)
    rg = self._ragged(want_pack=True)
    b, w = self.data.size()[:2]
    side = SideSpec(RIGHT if self._right_aligned else LEFT, width=w, rows=b * w)
    y, fin = _native.selective_scan(self.data.flatten(0, 1), delta.flatten(0, 1), A, B.flatten(0, 1), C.flatten(0, 1),
                                    initial, rg, side, reverse, want_final)
    return y.view(self.data.size()), fin


def _bind(cls, run):
    def selective_scan(self, delta: Tensor, A: Tensor, B: Tensor, C: Tensor, initial: Optional[Tensor] = None,
                       reverse: bool = False, return_final_state: bool = False):
        """per-sequence selective scan along time (see ``torchrua_b200.ssm``) -> a sequence of the same kind with the
        same metadata, or ``(it, final)`` with ``return_final_state``."""
        y, fin = run(self, delta, A, B, C, initial, reverse, return_final_state)
        out = self._replace(data=y)
        return (out, fin) if return_final_state else out

    cls.selective_scan = selective_scan


_bind(layout.C, _flat)
_bind(layout.P, _flat)
_bind(layout.L, _padded)
_bind(layout.R, _padded)
