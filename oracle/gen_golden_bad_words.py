"""Golden vectors of bad_words_ids: runs the installed transformers ``NoBadWordsLogitsProcessor`` on seeded cases and pins
oracle/decode_args.py's restatement of 4.16.2 on it.

The two agree bit for bit except where a sequence of L ids has L - 1 == cur_len and its first L - 1 ids are the whole decoder input:
4.16.2 bans its last id there, the installed 5.x (through ``SequenceBiasLogitsProcessor``, which skips L > cur_len) does not.  This
script asserts that the restatement equals HF's output with exactly those ids set to -inf, and that the seeded cases contain such rows.

Writes tests/golden/bad_words.npz: per case ``{name}_scores`` fp32 [rows, V], ``{name}_ids`` int64 [rows, cur_len] (decoder inputs
without [SEP]), ``{name}_words`` int32 (the sequences concatenated, each closed by -1) and ``{name}_out`` (the restatement's result).

    python -m oracle.gen_golden_bad_words
"""
from __future__ import annotations

import os

import numpy as np
import torch

from . import decode_args as DA

EOS = 102
OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "bad_words.npz")


def cases():
    """(name, scores [rows, V], ids [rows, cur_len], bad_words_ids) on a small alphabet so that sequence prefixes match the tails."""
    g = torch.Generator().manual_seed(20261022)
    V = 400
    out = []
    for i, (rows, cur_len) in enumerate([(4, 1), (4, 2), (6, 3), (6, 5), (8, 9), (5, 17), (3, 40), (4, 63)]):
        scores = torch.randn(rows, V, generator=g) * 3.0
        scores[0, 7] = -float("inf")                                   # -inf stays -inf
        ids = torch.randint(300, 306, (rows, cur_len), generator=g)
        ids[:, 0] = 101
        words = [[int(torch.randint(0, V, (1,), generator=g))] for _ in range(3)] + [[EOS], [EOS, 5], [7]]
        for r in range(rows):                                          # sequences that continue a row's tail, of every length up to d
            m = int(torch.randint(1, min(cur_len, 6) + 1, (1,), generator=g))
            words.append(ids[r, cur_len - m:].tolist() + [int(torch.randint(0, V, (1,), generator=g))])
        words.append(ids[0].tolist() + [11])                           # L - 1 == cur_len: the 4.16.2 / 5.x difference
        words.append([300, 301, 302, 13])                              # may or may not match
        words.append(ids[-1].tolist()[-1:] + [EOS])                    # a longer sequence may end in [SEP]
        if cur_len + 2 <= DA.MAX_LEN:
            words.append([101] + ids[1].tolist() + [17])               # longer than d + 1: never matches
        out.append((f"case{i}", scores, ids, words))
    return out


def flat(words):
    return np.array([w for s in words for w in list(s) + [-1]], dtype=np.int32)


def hf_apply(scores, ids, words):
    from transformers import NoBadWordsLogitsProcessor
    return NoBadWordsLogitsProcessor(words, eos_token_id=EOS)(ids, scores.clone())


def main():
    arrays, differing = {}, 0
    for name, scores, ids, words in cases():
        ours = DA.apply_bad_words(scores, ids.tolist(), words)
        ref = hf_apply(scores, ids, words)
        cur_len = ids.shape[1]
        expect = ref.clone()
        for r in range(ids.shape[0]):
            for w in words:
                if w != [EOS] and len(w) - 1 == cur_len and ids[r].tolist() == w[:-1]:
                    expect[r, w[-1]] = -float("inf")
                    differing += int(ref[r, w[-1]] != -float("inf"))
        assert torch.equal(ours, expect), name
        arrays.update({f"{name}_scores": scores.numpy(), f"{name}_ids": ids.numpy(), f"{name}_words": flat(words),
                       f"{name}_out": ours.numpy()})
    assert differing >= 4, differing
    np.savez_compressed(OUT, **arrays)
    print(f"wrote {OUT}: {len(arrays) // 4} cases, {differing} bans where 4.16.2 and the installed transformers differ")


if __name__ == "__main__":
    main()
