"""Per-sequence linear-chain CRF: log-partition, log-likelihood and Viterbi decode, for sequence labelling (NER, POS,
chunking, segmentation) on top of an encoder.  The reference has no counterpart; without it a user pads
(``x.left(0)``) and runs the forward algorithm as a Python loop over ``T`` that builds a ``(B, K, K)`` temporary per
step, all ``T`` of which autograd keeps.

Emissions hold one row of ``K`` tag scores per token ``(i, t)``: ``(N, K)`` for C and P, ``(B, W, K)`` for L and R.
``transitions[a, b]`` (``(K, K)``) scores tag ``a`` at ``t - 1`` followed by tag ``b`` at ``t``; ``start`` and ``end``
(``(K,)``) may be None, which means 0.  For a tag path ``y`` of sequence ``i`` with length ``len_i``::

    score(y) = start[y_0] + sum_t x(i, t)[y_t] + sum_{t>=1} transitions[y_{t-1}, y_t] + end[y_{len-1}]
    log Z_i  = logsumexp over all K^len paths of score(y)

* ``1 <= K <= 64``; ``transitions``, ``start`` and ``end`` have the emissions' dtype (fp32, fp64, fp16 or bf16).
* Accumulation is fp32 (fp64 for fp64).  Unlike the other ops of this package, the per-sequence outputs are returned in
  the ACCUMULATOR dtype -- fp32 for 16-bit emissions -- because a ``log Z`` of order 1e3 has a bf16 spacing of 4-8,
  which is useless as a loss.  ``strict_reductions()`` does not apply.
* Outputs are ``(B,)`` in ``token_sizes`` order (for P the original sequence index).
* An empty sequence has ``log Z = 0``, log-likelihood 0, decode score 0 and zero gradients.
* ``-inf`` in the emissions, ``transitions``, ``start`` or ``end`` forbids a tag or a transition (BIO constraints).  A
  sequence whose every path is forbidden has ``log Z = -inf`` and contributes zero gradient.  Behaviour is specified for
  inputs without NaN.
* A tag outside ``[0, K)`` at a token row is never dereferenced: that sequence's log-likelihood is NaN, the others are
  unaffected.  Tags at rows that hold no token are ignored, so ``-100`` padding is fine.
* Decode breaks ties toward the smallest tag index, for the predecessor at every step and for the last tag.  Rows that
  hold no token get ``-1``.
* The log-partition and the log-likelihood are once-differentiable (double backward raises); gradients reach the
  emissions, ``transitions``, ``start`` and ``end``, and the forward keeps its per-step state only when one is wanted.
  Marginals are the emission gradient of ``log Z``.  Decode has no gradient.
* Every result is bit-identical run to run and, for the same sequences, on C, L, P and R: each sequence runs on one warp
  of a fixed grid, in a fixed longest-first order.

One set of native kernels (rua_crf_forward / rua_crf_backward / rua_crf_decode) serves every layout, reading the rows
where they lie.
"""
from typing import Optional, Tuple

from torch import Tensor

from torchrua_b200 import _native
from torchrua_b200._lib import CAT, LEFT, PACK, RIGHT
from torchrua_b200._native import SideSpec
from torchrua_b200.layout import C, L, P, R

__all__ = ['segment_crf_log_partition', 'segment_crf_log_likelihood', 'segment_crf_decode']


def segment_crf_log_partition(emissions: Tensor, segment_sizes: Tensor, transitions: Tensor,
                              start: Optional[Tensor] = None, end: Optional[Tensor] = None) -> Tensor:
    """log Z of every segment of ``emissions`` (N, K) in C order; ``segment_sizes`` (S,) int64 -> (S,)."""
    _native.crf_check(emissions, transitions, start, end, 1)
    _native.require_cuda(segment_sizes)
    rg = _native.ragged_from_lengths(segment_sizes, want_pack=True)
    return _native.segment_crf(emissions, None, transitions, start, end, rg, SideSpec(CAT, rows=emissions.size()[0]))


def segment_crf_log_likelihood(emissions: Tensor, segment_sizes: Tensor, tags: Tensor, transitions: Tensor,
                               start: Optional[Tensor] = None, end: Optional[Tensor] = None) -> Tensor:
    """score(tags) - log Z of every segment -> (S,); ``tags`` (N,) int64, laid out like the emission rows."""
    _native.crf_check(emissions, transitions, start, end, 1, tags)
    _native.require_cuda(segment_sizes)
    rg = _native.ragged_from_lengths(segment_sizes, want_pack=True)
    return _native.segment_crf(emissions, tags, transitions, start, end, rg, SideSpec(CAT, rows=emissions.size()[0]))


def segment_crf_decode(emissions: Tensor, segment_sizes: Tensor, transitions: Tensor, start: Optional[Tensor] = None,
                       end: Optional[Tensor] = None) -> Tuple[Tensor, Tensor]:
    """Viterbi path of every segment: (tags (N,) int64, -1 past ``sum(segment_sizes)``; best score (S,))."""
    _native.crf_check(emissions, transitions, start, end, 1)
    _native.require_cuda(segment_sizes)
    rg = _native.ragged_from_lengths(segment_sizes, want_pack=True)
    return _native.crf_decode(emissions, transitions, start, end, rg, SideSpec(CAT, rows=emissions.size()[0]))


# ---------------------------------------------------------------------------------------------------------------------
# methods on the four layouts: the CRF runs on the flattened storage; decode keeps the layout and the metadata
# ---------------------------------------------------------------------------------------------------------------------
def _flat(self, tags: Optional[Tensor], transitions: Tensor, start: Optional[Tensor], end: Optional[Tensor]):
    """C / P: ``data`` is (N, K) -> (flat emissions, flat tags, ragged, side)."""
    _native.crf_check(self.data, transitions, start, end, 1, tags)
    cat = isinstance(self, C)
    rg = self._ragged(want_pack=True) if cat else self._ragged()
    return self.data, tags, rg, SideSpec(CAT if cat else PACK, rows=self.data.size()[0])


def _padded(self, tags: Optional[Tensor], transitions: Tensor, start: Optional[Tensor], end: Optional[Tensor]):
    """L / R: ``data`` is (B, W, K)."""
    _native.crf_check(self.data, transitions, start, end, 2, tags)
    rg = self._ragged(want_pack=True)
    b, w = self.data.size()[:2]
    side = SideSpec(RIGHT if self._right_aligned else LEFT, width=w, rows=b * w)
    flat_tags = None if tags is None else tags.flatten(start_dim=0, end_dim=1)
    return self.data.flatten(start_dim=0, end_dim=1), flat_tags, rg, side


def _bind(cls, run):
    def crf_log_partition(self, transitions: Tensor, start: Optional[Tensor] = None, end: Optional[Tensor] = None):
        """log Z of every sequence, (B,) in the accumulator dtype (see ``torchrua_b200.crf``)."""
        x, _, rg, side = run(self, None, transitions, start, end)
        return _native.segment_crf(x, None, transitions, start, end, rg, side)

    def crf_log_likelihood(self, tags: Tensor, transitions: Tensor, start: Optional[Tensor] = None,
                           end: Optional[Tensor] = None):
        """score(tags) - log Z of every sequence, (B,); ``tags`` int64 laid out like ``data`` without its tag
        dimension (rows that hold no token are ignored)."""
        x, flat_tags, rg, side = run(self, tags, transitions, start, end)
        return _native.segment_crf(x, flat_tags, transitions, start, end, rg, side)

    def crf_decode(self, transitions: Tensor, start: Optional[Tensor] = None, end: Optional[Tensor] = None):
        """(Viterbi tags in the same layout and metadata, int64 with -1 at rows that hold no token; best scores (B,))."""
        x, _, rg, side = run(self, None, transitions, start, end)
        tags, best = _native.crf_decode(x, transitions, start, end, rg, side)
        return self._replace(data=tags.view(self.data.shape[:-1])), best

    for fn in (crf_log_partition, crf_log_likelihood, crf_decode):
        setattr(cls, fn.__name__, fn)


_bind(C, _flat)
_bind(P, _flat)
_bind(L, _padded)
_bind(R, _padded)
