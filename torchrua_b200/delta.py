"""Per-sequence gated delta rule (Gated DeltaNet), the linear-attention mixer of current hybrid models: a scalar log
decay ``g`` and a write strength ``beta`` per token and value head, a ``(K, V)`` state per value head, and ``q`` / ``k``
shared by the value heads of a key group.  The reference has no counterpart; without it a user pads every sequence to
``T`` and runs a chunked form that materialises ``(B, chunks, Q, Q, H)`` tensors, or hands the C storage's offsets to a
Triton library.

For token ``(i, t)``, value head ``h < H`` and key group ``c = h // (H / G)``, with ``S`` the ``(K, V)`` state of head
``h`` (the ``naive_recurrent_gated_delta_rule`` of flash-linear-attention, state order ``(K, V)``)::

    S'_t        = exp(g_t[h]) * S_(t-1)                                S_(-1) = initial[i, h] (0 without one)
    u_t         = beta_t[h] * (v_t[h] - S'_t^T k_t[c])
    S_t         = S'_t + k_t[c] (outer) u_t
    o_t[h]      = scale * S_t^T q_t[c]                                 scale = K ** -0.5 when None
    final[i, h] = S at the last token (initial[i, h], or 0, for an empty sequence)

``reverse=True`` runs from each sequence's end: ``S_t`` depends on ``S_(t+1)``, ``S_(len_i) = initial[i]`` and
``final[i]`` is the state at ``t = 0`` (the convention of ``linear_recurrence``, ``selective_scan`` and ``ssd``).

* ``v`` is ``(rows, H, V)`` (``(B, W, H, V)`` for L and R), ``q`` and ``k`` are ``(rows, G, K)`` with ``H % G == 0``,
  ``g`` and ``beta`` are ``(rows, H)``, all in the payload's layout.  ``v``, ``q``, ``k`` and ``beta`` share one dtype:
  fp16, bf16, fp32 or fp64.
* ``g``, ``initial`` and ``final`` are in the ACCUMULATOR dtype: fp32, or fp64 for fp64 payloads (``g`` is the log decay
  as the model computes it in fp32).  ``initial`` and ``final`` are ``(batch, H, K, V)`` in ``token_sizes`` order (for
  P the original sequence index).
* ``1 <= K <= 128`` and ``1 <= V <= 256``.
* Rows that hold no token (L / R padding, C rows past ``sum(sizes)``) are copied through from ``v``; there the ``v``
  gradient passes ``grad_out`` through and the ``q``, ``k``, ``g`` and ``beta`` gradients are 0.
* Gradients reach ``v``, ``q``, ``k``, ``g``, ``beta`` and ``initial``; an unwanted one is not written.  The forward
  keeps nothing for the backward, which recomputes the states it needs.  ``final`` is not differentiable.  Double
  backward raises.
* Every result is bit-identical run to run and, for the same sequences, on C, L, P and R: no float atomics, and every
  sum runs in a fixed order.

Precision.  Each sequence is cut into chunks of its own tokens (64 for fp16 / bf16, 32 for fp32, 16 for fp64), and within
a chunk the rule is a few small matrix products, on tensor cores for fp16 / bf16, around the chunk's WY / UT transform
``T = (I + strict_tril(diag(beta) (K K^T) o exp(cum_t - cum_s)))^-1``:

* the carried state and its adjoint are always kept in the accumulator type and never rounded between chunks;
* ``T``, the in-chunk cumulative log decay and every exponential are computed in the accumulator type, the decays
  always as ``exp(cum_t - cum_s)``;
* for 16-bit payloads each operand of a tensor-core product is rounded to the payload dtype once (among them ``T``, the
  decay-masked scores, the corrected values ``V'`` and the copy of the state that ``q`` and ``k`` read), with fp32
  accumulation;
* fp32 and fp64 payloads round nothing but the output.

Out of scope: the L2 norm of ``q`` / ``k``, the gate activation ``-exp(A_log) * softplus(a + dt_bias)``, the output
gate and norm (pointwise: write them in torch), ``K > 128``, ``V > 256``, a gradient through ``final``, channel-wise
gates (KDA), several Householder factors per token (DeltaProduct), a port of the products to tcgen05, and speed for
single-token decode steps (they work: ``len = 1`` sequences with ``initial``).

One set of native kernels (rua_gdn_forward / rua_gdn_backward) serves every layout, reading the rows where they lie.
"""
from typing import Optional

from torch import Tensor

from torchrua_b200 import _native
from torchrua_b200 import layout
from torchrua_b200._lib import CAT, LEFT, PACK, RIGHT
from torchrua_b200._native import SideSpec

__all__ = ['segment_gated_delta_rule']


def segment_gated_delta_rule(tensor: Tensor, segment_sizes: Tensor, q: Tensor, k: Tensor, g: Tensor, beta: Tensor,
                             scale: Optional[float] = None, initial: Optional[Tensor] = None, reverse: bool = False,
                             return_final_state: bool = False):
    """gated delta rule along every segment of ``tensor`` = v (rows, H, V) in C order; ``segment_sizes`` (S,) int64,
    ``q`` and ``k`` (rows, G, K), ``g`` and ``beta`` (rows, H), ``initial`` (S, H, K, V) or None -> o, or
    ``(o, final)`` with ``return_final_state``."""
    _, _, K, _ = _native.gdn_check(tensor, q, k, g, beta, initial, segment_sizes.shape[0], 1)
    _native.require_cuda(segment_sizes)
    rg = _native.ragged_from_lengths(segment_sizes, want_pack=True)
    o, fin = _native.gdn(tensor, q, k, g, beta, initial, _native.gdn_scale(scale, K), rg,
                         SideSpec(CAT, rows=tensor.size()[0]), reverse, return_final_state)
    return (o, fin) if return_final_state else o


# ---------------------------------------------------------------------------------------------------------------------
# methods on the four layouts: the rule runs on the flattened storage, the result keeps the layout and the metadata
# ---------------------------------------------------------------------------------------------------------------------
def _batch(self) -> int:
    if isinstance(self, layout.C):
        return self.token_sizes.shape[0]
    if self.unsorted_indices is not None:
        return self.unsorted_indices.numel()
    return int(self.batch_sizes[0]) if self.batch_sizes.numel() else 0


def _flat(self, q, k, g, beta, scale, initial, reverse, want_final):
    """C / P: ``data`` is (rows, H, V)."""
    _, _, K, _ = _native.gdn_check(self.data, q, k, g, beta, initial, _batch(self), 1)
    cat = isinstance(self, layout.C)
    rg = self._ragged(want_pack=True) if cat else self._ragged()
    side = SideSpec(CAT if cat else PACK, rows=self.data.size()[0])
    return _native.gdn(self.data, q, k, g, beta, initial, _native.gdn_scale(scale, K), rg, side, reverse, want_final)


def _padded(self, q, k, g, beta, scale, initial, reverse, want_final):
    """L / R: ``data`` is (B, W, H, V); q, k, g and beta at padding positions are ignored."""
    _, _, K, _ = _native.gdn_check(self.data, q, k, g, beta, initial, self.data.shape[0], 2)
    rg = self._ragged(want_pack=True)
    b, w = self.data.size()[:2]
    side = SideSpec(RIGHT if self._right_aligned else LEFT, width=w, rows=b * w)
    o, fin = _native.gdn(self.data.flatten(0, 1), q.flatten(0, 1), k.flatten(0, 1), g.flatten(0, 1),
                         beta.flatten(0, 1), initial, _native.gdn_scale(scale, K), rg, side, reverse, want_final)
    return o.view(self.data.size()), fin


def _bind(cls, run):
    def gated_delta_rule(self, q: Tensor, k: Tensor, g: Tensor, beta: Tensor, scale: Optional[float] = None,
                         initial: Optional[Tensor] = None, reverse: bool = False, return_final_state: bool = False):
        """per-sequence gated delta rule along time with this sequence as v (see ``torchrua_b200.delta``) -> a
        sequence of the same kind with the same metadata, or ``(it, final)`` with ``return_final_state``."""
        o, fin = run(self, q, k, g, beta, scale, initial, reverse, return_final_state)
        out = self._replace(data=o)
        return (out, fin) if return_final_state else out

    cls.gated_delta_rule = gated_delta_rule


_bind(layout.C, _flat)
_bind(layout.P, _flat)
_bind(layout.L, _padded)
_bind(layout.R, _padded)
