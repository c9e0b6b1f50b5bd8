"""TEST INFRASTRUCTURE ONLY - beam search with question-history n-gram blocking (plain PyTorch / Python, CPU).

Extends the beam contract of ``oracle/beam.py`` with the reference's n-gram blocking (utils/decoding_utils.py:38-78, applied
to the questioner with n = 4, generate.py:124).  The reference has no beam search, so the combination is defined here the way
``transformers==4.16.2`` ``beam_search`` runs a logits processor: on the log-softmax scores, before the beam scores are added.

Arithmetic contract (on top of oracle/beam.py's, which is unchanged):
  * at step t the key of beam k of image b is its decoded prefix [CLS] + tokens[b, k, :t]; its banned set is exactly
    ``restatement.ngram_banned_tokens(hist_b, key, n)`` with hist_b = enc_input_ids[b] * (enc_segments[b] == 0)
  * logZ is computed over the full, unbanned row, exactly as in oracle/beam.py
  * candidate score = fp32(fp32(x - logZ) + beam_score); banned (beam, token) pairs are set to -inf before the top-2K
    (log_softmax, then the processor, then the beam score; no renormalisation)
  * everything else (tie order, EOS handling, hypothesis scores, ``done``) is oracle/beam.py's
With n = 0 nothing is banned and the results are those of oracle/beam.py (tests/test_beam_ngram.py checks it).
"""
from __future__ import annotations

import torch

from . import restatement as R
from .beam import EOS, BeamState, candidate_scores, top_candidates


def question_history(enc_input_ids: torch.Tensor, enc_segments: torch.Tensor):
    """Per-image question history as lists: ids * (segments == 0) (models/visual_dialog_model.py:98-99)."""
    return (enc_input_ids * (enc_segments == 0).long()).tolist()


class BlockedBeamState(BeamState):
    """``BeamState`` whose ``step`` also takes the n-gram blocking size and the per-image question history."""

    def banned(self, hist, n: int):
        """List over the B*K beam rows of the tokens banned at the current step."""
        out = []
        for b in range(self.B):
            for k in range(self.K):
                key = [R.CLS] + self.tokens[b, k, : self.t].tolist()
                out.append(R.ngram_banned_tokens(hist[b], key, n) if n > 0 else [])
        return out

    def step(self, logits: torch.Tensor, ngram_blocking_size: int = 0, hist=None):
        """One ``beam_search`` iteration on logits [B*K, V]; ``hist``: per-image question history (``question_history``),
        needed when ``ngram_blocking_size`` > 0."""
        B, K, V = self.B, self.K, self.V
        cur_len = self.t + 1
        sc = candidate_scores(logits.float(), self.beam_scores)
        if ngram_blocking_size > 0:
            for row, toks in enumerate(self.banned(hist, ngram_blocking_size)):
                b, k = divmod(row, K)
                for w in toks:
                    sc[b, k * V + w] = -float("inf")
        val, idx = top_candidates(sc, 2 * K)
        # from here on: BeamState.step verbatim
        nb_scores = torch.zeros(B, K, dtype=torch.float32)
        nb_tokens = torch.zeros(B, K, dtype=torch.int64)
        nb_idx = torch.zeros(B, K, dtype=torch.int64)
        for b in range(B):
            if self.done[b]:
                continue
            n = 0
            for rank in range(2 * K):
                flat = int(idx[b, rank]); beam, tok = flat // V, flat % V
                s = val[b, rank]
                if tok == EOS:
                    if rank >= K:
                        continue
                    self._add(b, self.tokens[b, beam, : self.t].tolist(), s.item(), cur_len)
                else:
                    nb_scores[b, n] = s; nb_tokens[b, n] = tok; nb_idx[b, n] = beam
                    n += 1
                if n == K:
                    break
            assert n == K
            if len(self.hyps[b]) >= K:
                cur = float(val[b].max().item()) / float(cur_len)
                if self.worst[b] >= cur:
                    self.done[b] = True
        new_tokens = self.tokens.gather(1, nb_idx[:, :, None].expand(-1, -1, self.T)).clone()
        new_tokens[:, :, self.t] = nb_tokens
        self.tokens = new_tokens
        self.beam_scores = nb_scores
        self.last_beam_idx, self.last_tokens = nb_idx, nb_tokens
        self.t += 1
        return nb_idx, nb_tokens, nb_scores


def beam_search(sd, enc_cfg, dec_cfg, batch, num_beams=5, max_new=18, ngram_blocking_size=0, precomputed_encoder=None):
    """oracle/beam.py:beam_search with n-gram blocking against the question history of ``batch``."""
    ids, seg, att = batch["enc_input_ids"], batch["enc_segments"], batch["enc_att_mask"]
    B, K = ids.shape[0], num_beams
    if precomputed_encoder is not None:
        seq_t, seq_v = precomputed_encoder
    else:
        seq_t, seq_v = R.encoder(sd, enc_cfg, ids, batch["enc_image_feat"], batch["enc_image_loc"], seg, att, batch["enc_image_mask"])
    enc_h, enc_m = R.vlfusion(sd, seq_t, seq_v, att, batch["enc_image_mask"])
    enc_h = enc_h.repeat_interleave(K, 0); enc_m = enc_m.repeat_interleave(K, 0)
    hist = question_history(ids, seg)
    st = BlockedBeamState(B, K, dec_cfg.vocab_size, max_new)
    for t in range(max_new):
        prefix = torch.cat((torch.full((B * K, 1), R.CLS, dtype=torch.int64), st.tokens.reshape(B * K, -1)[:, :t]), 1)
        h = R.decoder_hidden(sd, dec_cfg, prefix, None, enc_h, enc_m)
        st.step(R.lm_logits(sd, h[:, -1]), ngram_blocking_size, hist)
        if bool(st.done.all()):
            break
    return st.finalize()


def banned_ngrams(hist, n: int):
    """The set of n-grams (tuples) of one history row that blocking bans: those without a special id."""
    return {tuple(hist[i:i + n]) for i in range(len(hist) - n + 1) if not set(hist[i:i + n]) & set(R.SPECIAL_IDS)}


def contains_banned_ngram(hist, seq, n: int) -> bool:
    """True when [CLS] + seq holds an n-gram of ``hist`` that blocking would have banned."""
    toks = [R.CLS] + [int(x) for x in seq]
    bad = banned_ngrams(hist, n)
    return any(tuple(toks[i:i + n]) in bad for i in range(len(toks) - n + 1))
