"""TEST INFRASTRUCTURE ONLY - pins oracle/processors.py on HF's own logits processors and writes tests/golden/logits_processors.npz.

Runs the installed ``transformers`` ``RepetitionPenaltyLogitsProcessor``, ``NoRepeatNGramLogitsProcessor`` and
``MinLengthLogitsProcessor`` on seeded cases and asserts that the restatement gives the same scores, bit for bit.  For 2-D scores
(``[rows, V]``) the code these classes run is the one of transformers 4.16.2, the reference's pin: the gather / where / scatter of the
repetition penalty, ``_get_ngrams`` / ``_get_generated_ngrams`` / ``_calc_banned_ngram_tokens`` (cur_len + 1 < n bans nothing), and
-inf on the eos id while ``input_ids.shape[-1] < min_length``.  (The 3-D paths and ``prompt_ignore_length`` that later versions added
are not used.)

Cases: ids that repeat in a row, positive / negative / -inf scores, n = 1 and n longer than the decoder input, cur_len on both sides
of m, all three processors together.  Usage: ``python -m oracle.gen_golden_processors`` (needs transformers).
"""
from __future__ import annotations

import os

import numpy as np
import torch

from . import processors as LP

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "logits_processors.npz")
V = 120


def cases():
    """(name, scores [rows, V] fp32, input_ids [rows, L] int64, p, n, m) with seeded contents."""
    g = torch.Generator().manual_seed(20261022)
    out = []
    for ci, (L, p, n, m) in enumerate([(1, 1.3, 0, 0), (6, 1.3, 0, 0), (9, 0.7, 0, 0), (12, 2.0, 0, 0),
                                       (8, 1.0, 1, 0), (8, 1.0, 2, 0), (10, 1.0, 3, 0), (5, 1.0, 7, 0), (4, 1.0, 5, 0),
                                       (5, 1.0, 0, 5), (5, 1.0, 0, 6), (6, 1.0, 0, 6), (1, 1.0, 0, 3),
                                       (11, 1.5, 2, 14), (7, 0.8, 3, 7), (16, 1.2, 4, 20)]):
        rows = 6
        s = torch.randn(rows, V, generator=g) * 4.0
        s[torch.rand(rows, V, generator=g) < 0.05] = -float("inf")
        s[:, 102] = torch.randn(rows, generator=g) * 4.0
        s[0, :] = s[0, :].abs()                                                  # a row of positive scores
        s[1, :] = -s[1, :].abs()                                                 # a row of negative scores
        # small alphabets so that ids and n-grams repeat; row 5 cycles a 2-gram; a few rows carry -inf ids
        ids = torch.randint(3, 3 + max(2, L // 3), (rows, L), generator=g)
        ids[5] = torch.tensor([7, 8] * L)[:L]
        ids[4, 0] = 101
        s[2, ids[2, 0]] = -float("inf")
        out.append((f"case{ci}", s.float(), ids.long(), p, n, m))
    return out


def hf_apply(scores, ids, p, n, m):
    from transformers.generation.logits_process import (MinLengthLogitsProcessor, NoRepeatNGramLogitsProcessor,
                                                        RepetitionPenaltyLogitsProcessor)
    out = scores.clone()
    if p != 1.0:
        out = RepetitionPenaltyLogitsProcessor(penalty=p)(ids, out)
    if n > 0:
        out = NoRepeatNGramLogitsProcessor(n)(ids, out)
    if m > 0:
        out = MinLengthLogitsProcessor(m, eos_token_id=102)(ids, out)
    return out


def main():
    arrays = {}
    for name, s, ids, p, n, m in cases():
        hf = hf_apply(s, ids, p, n, m)
        ours = LP.apply(s, ids.tolist(), repetition_penalty=p, no_repeat_ngram_size=n, min_length=m)
        assert torch.equal(torch.isinf(hf), torch.isinf(ours)) and torch.equal(hf[~torch.isinf(hf)], ours[~torch.isinf(ours)]), name
        assert torch.equal(hf, ours), name
        arrays[f"{name}_scores"] = s.numpy()
        arrays[f"{name}_ids"] = ids.numpy()
        arrays[f"{name}_params"] = np.array([p, n, m], dtype=np.float64)
        arrays[f"{name}_out"] = hf.numpy()
    np.savez_compressed(OUT, **arrays)
    print(f"{OUT}: {len(arrays) // 4} cases, {os.path.getsize(OUT)} bytes")


if __name__ == "__main__":
    main()
