"""TEST INFRASTRUCTURE ONLY - N-best beam finalisation (``num_return_sequences``), plain Python, CPU.

``transformers==4.16.2`` ``BeamSearchScorer.finalize`` with ``num_return_sequences = N``: the unfinished beams of an image are added
to its hypotheses as for N = 1, then the hypotheses - kept in insertion order - are sorted by score with a STABLE ascending sort and
``pop()``-ed N times.  So output n of an image is its hypothesis of rank n by (score descending, insertion order descending): among
equal scores the later-inserted hypothesis comes first.  Each gets [SEP] appended when it fits, like ``BeamState.finalize``.  Rows
are image-major (row b*N + n).

Works on ``oracle/beam.py:BeamState``, ``oracle/beam_ngram.py:BlockedBeamState`` and any subclass whose decoder input is ``P``
tokens long (attribute ``P``; the [CLS] start is P = 1), such as the prefix beam state of tests/test_decoder_prefix.py.  With
N = 1 it is the state's own ``finalize``.
"""
from __future__ import annotations

import torch

from .beam import EOS


def pop_order(hyps, N):
    """The first N of ``hyps`` (list of (score, tokens) in insertion order) in ``sorted(...).pop()`` order."""
    srt = sorted(hyps, key=lambda x: x[0])           # stable: insertion order among equal scores
    return [srt.pop() for _ in range(N)]


def finalize_nbest(st, N):
    """``st.finalize()`` returning the N best hypotheses per image: (sequences [B*N, T] int64, scores [B*N] fp64)."""
    B, K, T = st.B, st.K, st.T
    if not 1 <= N <= K:
        raise ValueError(f"num_return_sequences must be in 1..num_beams ({K}), got {N}")
    P = getattr(st, "P", 1)
    seq = torch.zeros(B * N, T, dtype=torch.int64)
    scores = torch.zeros(B * N, dtype=torch.float64)
    for b in range(B):
        if not st.done[b]:
            for k in range(K):
                st._add(b, st.tokens[b, k, : st.t].tolist(), st.beam_scores[b, k].item(), st.t + P)
        for n, (score, toks) in enumerate(pop_order(st.hyps[b], N)):
            row = b * N + n
            seq[row, : len(toks)] = torch.tensor(toks, dtype=torch.int64)
            if len(toks) < T:
                seq[row, len(toks)] = EOS
            scores[row] = score
    return seq, scores
