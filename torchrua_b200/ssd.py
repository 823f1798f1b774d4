"""Per-sequence Mamba-2 (SSD) state-space scan, the sequence mixer of current hybrid models: a scalar decay per head,
a ``(P, N)`` state per head, and ``B`` / ``C`` shared by the heads of a group.  The reference has no counterpart;
without it a user pads every sequence to ``T`` and runs a chunked einsum that materialises ``(B, chunks, Q, Q, H)``
decay tensors, or scans the C storage with a dense-batch kernel, which leaks state from one sequence into the next.

For token ``(i, t)``, head ``h < H``, head channel ``p < P``, state ``n < N`` and group ``g(h) = h // (H / G)``::

    dA_t        = exp(delta_t[h] * A[h])                                           (a scalar per token and head)
    h_t[p, n]   = dA_t * h_(t-1)[p, n] + delta_t[h] * x_t[h, p] * B_t[g, n],     h_(-1) = initial[i, h] (0 without one)
    y_t[h, p]   = sum_n C_t[g, n] * h_t[p, n]
    final[i, h] = h at the last token (initial[i, h], or 0, for an empty sequence)

``reverse=True`` runs from each sequence's end: ``h_t`` depends on ``h_(t+1)``, ``h_(len_i) = initial[i]`` and
``final[i]`` is the state at ``t = 0`` (the convention of ``linear_recurrence`` and ``selective_scan``).

* ``x`` is ``(rows, H, P)`` (``(B, W, H, P)`` for L and R), ``delta`` is ``(rows, H)``, ``B`` and ``C`` are
  ``(rows, G, N)`` with ``H % G == 0``, all in the payload's layout.  ``x``, ``delta``, ``B`` and ``C`` share one dtype:
  fp16, bf16, fp32 or fp64.
* ``A`` is ``(H,)``; ``initial`` and ``final`` are ``(batch, H, P, N)`` (Mamba-2's state order) in ``token_sizes`` order
  (for P the original sequence index).  All three are in the ACCUMULATOR dtype: fp32, or fp64 for fp64 payloads.
* ``1 <= P <= 64`` and ``1 <= N <= 128``.
* Rows that hold no token (L / R padding, C rows past ``sum(sizes)``) are copied through from ``x``; there the ``x``
  gradient passes ``grad_out`` through and the ``delta``, ``B`` and ``C`` gradients are 0.
* Gradients reach ``x``, ``delta``, ``A``, ``B``, ``C`` and ``initial`` (0 for an empty sequence); an unwanted one is not
  written.  The forward keeps nothing for the backward, which recomputes the states it needs, so its memory and time
  are the same with and without autograd.  ``final`` is not differentiable.  Double backward raises.
* Every result is bit-identical run to run and, for the same sequences, on C, L, P and R: no float atomics, and every
  sum runs in a fixed order.

Precision.  Each sequence is cut into chunks of 64 of its tokens (16 for fp64), and within a chunk the scan is a few
small matrix products, on tensor cores for fp16 / bf16:

* the carried state is always kept in the accumulator type and never rounded between chunks;
* for 16-bit payloads the operands of the tensor-core products are rounded to the payload dtype once each: ``delta*x``,
  the decay-masked scores ``exp(cum_t - cum_s) * (C_t . B_s)``, the decay-weighted ``B`` of the state update and the copy
  of the state that ``C`` reads (Mamba-2's own kernels do the same), with fp32 accumulation;
* fp32 and fp64 payloads round nothing but the output.

Out of scope: ``softplus(delta + dt_bias)``, the ``D * x`` skip, the ``z`` gate and the norm (pointwise: write them in
torch), ``P > 64`` and ``N > 128``, a gradient through ``final``, a port of the products to tcgen05, and speed for
single-token decode steps (they work: ``len = 1`` sequences with ``initial``).

One set of native kernels (rua_ssd_forward / rua_ssd_backward) serves every layout, reading the rows where they lie.
"""
from typing import Optional

from torch import Tensor

from torchrua_b200 import _native
from torchrua_b200 import layout
from torchrua_b200._lib import CAT, LEFT, PACK, RIGHT
from torchrua_b200._native import SideSpec

__all__ = ['segment_ssd']


def segment_ssd(tensor: Tensor, segment_sizes: Tensor, delta: Tensor, A: Tensor, B: Tensor, C: Tensor,
                initial: Optional[Tensor] = None, reverse: bool = False, return_final_state: bool = False):
    """SSD scan along every segment of ``tensor`` (rows, H, P) in C order; ``segment_sizes`` (S,) int64, ``delta``
    (rows, H), ``B`` and ``C`` (rows, G, N), ``A`` (H,), ``initial`` (S, H, P, N) or None -> y, or ``(y, final)`` with
    ``return_final_state``."""
    _native.ssd_check(tensor, delta, A, B, C, initial, segment_sizes.shape[0], 1)
    _native.require_cuda(segment_sizes)
    rg = _native.ragged_from_lengths(segment_sizes, want_pack=True)
    y, fin = _native.ssd(tensor, delta, A, B, C, initial, rg, SideSpec(CAT, rows=tensor.size()[0]), reverse,
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
    """C / P: ``data`` is (rows, H, P)."""
    _native.ssd_check(self.data, delta, A, B, C, initial, _batch(self), 1)
    cat = isinstance(self, layout.C)
    rg = self._ragged(want_pack=True) if cat else self._ragged()
    side = SideSpec(CAT if cat else PACK, rows=self.data.size()[0])
    return _native.ssd(self.data, delta, A, B, C, initial, rg, side, reverse, want_final)


def _padded(self, delta, A, B, C, initial, reverse, want_final):
    """L / R: ``data`` is (B, W, H, P); delta, B and C at padding positions are ignored."""
    _native.ssd_check(self.data, delta, A, B, C, initial, self.data.shape[0], 2)
    rg = self._ragged(want_pack=True)
    b, w = self.data.size()[:2]
    side = SideSpec(RIGHT if self._right_aligned else LEFT, width=w, rows=b * w)
    y, fin = _native.ssd(self.data.flatten(0, 1), delta.flatten(0, 1), A, B.flatten(0, 1), C.flatten(0, 1), initial,
                         rg, side, reverse, want_final)
    return y.view(self.data.size()), fin


def _bind(cls, run):
    def ssd(self, delta: Tensor, A: Tensor, B: Tensor, C: Tensor, initial: Optional[Tensor] = None,
            reverse: bool = False, return_final_state: bool = False):
        """per-sequence Mamba-2 (SSD) scan along time (see ``torchrua_b200.ssd``) -> a sequence of the same kind with
        the same metadata, or ``(it, final)`` with ``return_final_state``."""
        y, fin = run(self, delta, A, B, C, initial, reverse, return_final_state)
        out = self._replace(data=y)
        return (out, fin) if return_final_state else out

    cls.ssd = ssd


_bind(layout.C, _flat)
_bind(layout.P, _flat)
_bind(layout.L, _padded)
_bind(layout.R, _padded)
