"""TEST INFRASTRUCTURE ONLY - HF length_penalty / early_stopping of the beam modes and bad_words_ids in every mode (plain PyTorch /
Python, CPU).

Restates, as ``gstvd_generate`` applies them (include/gstvd.h), three ``generate()`` arguments of ``transformers==4.16.2`` (the
reference's pin):

``length_penalty`` lambda and ``early_stopping`` (``BeamHypotheses.add`` / ``is_done``, used by ``BeamSearchScorer`` in beam search,
group beam search and beam sampling).  lambda is the fp32 value the C struct holds, read as fp64.  len = a hypothesis's decoder-input
length: the image's prefix length P plus its generated tokens, without the closing [SEP] (P + t when it closes at step t):
  * a hypothesis scores fp64(sum_logprobs) / len ** lambda, the power being Python's float ** float (libm pow); lambda = 1 divides by len
    exactly as oracle/beam.py does, lambda = 0 does not normalise;
  * is_done(best_sum, cur_len): the heap holds num_beams hypotheses and (early_stopping, or worst_score >= best_sum / cur_len ** lambda);
  * finalisation (oracle/beam_nbest.py, unchanged) adds the unfinished beams through the same ``_add``, so the returned scores are the
    penalised ones (HF ``sequences_scores``).
Sampling ignores both.  transformers 5.x no longer has ``BeamSearchScorer``, so this part is an unpinned restatement, like the other beam
oracles.

``bad_words_ids`` (``NoBadWordsLogitsProcessor``), on a row's decoder input d (HF input_ids; [SEP] read as [PAD], oracle/processors.py)
with cur_len = len(d).  For a listed sequence w[0..L-1]:
  * L = 1: w[0] is -inf at every step;
  * L > 1: w[L-1] is -inf when L - 1 <= cur_len and d[-(L-1):] == w[:L-1] (4.16.2 ``_tokens_match``);
  * a sequence equal to [SEP] alone is dropped (HF filters ``[eos_token_id]``).
It acts where oracle/processors.py's processors act, and like two of them it only writes -inf.  The installed transformers 5.x implements
the processor through ``SequenceBiasLogitsProcessor``, which skips a sequence with L > cur_len: it differs from 4.16.2 exactly when
L - 1 == cur_len (the sequence's prefix covers the whole of d).  oracle/gen_golden_bad_words.py pins this file on the installed class
everywhere else, asserts that difference, and writes tests/golden/bad_words.npz.

The decode oracles below are those of oracle/processors.py with these arguments added; with the HF defaults (1.0, False, no list) every
step and the finalisation compute exactly what the oracle/processors.py states compute (tests/test_length_penalty.py checks it).
"""
from __future__ import annotations

import math

import numpy as np
import torch

from . import processors as LP
from . import restatement as R
from .beam import log_z, top_candidates
from .beam_sample import NSEL, candidate_seed, gumbel_keys, kept_count, uniforms
from .processors import ProcessedBeamSampleState, ProcessedGroupBeamState, _checked, _encoded

EOS, PAD = 102, 0
MAX_SEQS, MAX_LEN, MAX_IDS = 1024, 64, 4096          # the engine's limits of one list


def check_beam_args(length_penalty=1.0, early_stopping=False):
    if not math.isfinite(float(length_penalty)):
        raise ValueError(f"length_penalty must be finite, got {length_penalty}")
    if int(early_stopping) not in (0, 1):
        raise ValueError(f"early_stopping must be 0 / 1, got {early_stopping}")


def check_bad_words(bad_words_ids, vocab_size=None):
    """The engine's rule for a list: at most 1024 sequences of 1..64 ids, 4096 ids in all, ids in [0, vocab)."""
    seqs = [list(map(int, s)) for s in (bad_words_ids or [])]
    if len(seqs) > MAX_SEQS or sum(map(len, seqs)) > MAX_IDS:
        raise ValueError(f"at most {MAX_SEQS} bad-word sequences and {MAX_IDS} ids")
    for s in seqs:
        if not 1 <= len(s) <= MAX_LEN or any(w < 0 or (vocab_size is not None and w >= vocab_size) for w in s):
            raise ValueError(f"bad-word sequence {s}: 1..{MAX_LEN} ids in [0, vocab)")
    return seqs


def bad_words_banned(d, bad_words_ids):
    """The ids NoBadWordsLogitsProcessor (4.16.2) bans for one row with decoder input d (a list)."""
    out = []
    for w in bad_words_ids or []:
        w = [int(x) for x in w]
        if w == [EOS]:
            continue
        m = len(w) - 1
        if m <= len(d) and (m == 0 or list(d[len(d) - m:]) == w[:m]):
            out.append(w[-1])
    return out


def apply_bad_words(scores, d_rows, bad_words_ids):
    """bad_words_ids on scores [rows, V] fp32 (a new tensor); d_rows: per-row decoder inputs."""
    out = scores.float().clone()
    if not bad_words_ids:
        return out
    for r, d in enumerate(d_rows):
        banned = bad_words_banned([int(w) for w in d], bad_words_ids)
        if banned:
            out[r, torch.tensor(banned, dtype=torch.int64)] = -float("inf")
    return out


def apply(scores, d_rows, procs, bad_words_ids):
    """oracle/processors.py's processors, then the bad words (both only act on their own ids; the bans commute with them)."""
    return apply_bad_words(LP.apply(scores, d_rows, **procs), d_rows, bad_words_ids)


class _LengthPenalty:
    """BeamHypotheses.add / is_done with length_penalty and early_stopping, mixed into a beam state before its base class."""

    def _set_length_args(self, length_penalty, early_stopping):
        check_beam_args(length_penalty, early_stopping)
        self.length_penalty = float(np.float32(length_penalty))        # the fp32 the C struct holds
        self.early_stopping = bool(early_stopping)

    def _denom(self, length):
        return float(length) if self.length_penalty == 1.0 else float(length) ** self.length_penalty

    def _add(self, b, toks, sum_logprobs, length):
        score = float(sum_logprobs) / self._denom(length)
        h = self.hyps[b]
        if len(h) < self.K or score > self.worst[b]:
            h.append((score, list(toks)))
            if len(h) > self.K:
                srt = sorted([(s, i) for i, (s, _) in enumerate(h)])
                del h[srt[0][1]]
                self.worst[b] = srt[1][0]
            else:
                self.worst[b] = min(score, self.worst[b])

    def _is_done(self, b, best_sum, cur_len):
        if len(self.hyps[b]) < self.K:
            return False
        return self.early_stopping or self.worst[b] >= float(best_sum) / self._denom(cur_len)


class ArgsGroupBeamState(_LengthPenalty, ProcessedGroupBeamState):
    """ProcessedGroupBeamState (beam search with or without groups and a decoder prefix) with length_penalty, early_stopping and bad
    words.  Each step is the base step with the two marked lines changed."""

    def __init__(self, B, K, V, max_new=18, num_beam_groups=1, diversity_penalty=0.0, prefix=None, processors=None, length_penalty=1.0,
                 early_stopping=False, bad_words_ids=None):
        super().__init__(B, K, V, max_new, num_beam_groups, diversity_penalty, prefix, processors)
        self._set_length_args(length_penalty, early_stopping)
        self.bad_words = check_bad_words(bad_words_ids, V)

    def step(self, logits, ngram_blocking_size=0, hist=None):
        B, K, V, G, gs = self.B, self.K, self.V, self.G, self.gs
        cur_len = self.t + self.P
        lg = logits.float()
        lp = (lg - log_z(lg)).reshape(B, K, V)
        if ngram_blocking_size > 0:
            for row, toks in enumerate(self.banned(hist, ngram_blocking_size)):
                b, k = divmod(row, K)
                for w in toks:
                    lp[b, k, w] = -float("inf")
        d_rows = self.decoder_inputs()
        nb_scores = torch.zeros(B, K, dtype=torch.float32)
        nb_tokens = torch.zeros(B, K, dtype=torch.int64)
        nb_idx = torch.zeros(B, K, dtype=torch.int64)
        for b in range(B):
            for g in range(G):
                lo = g * gs
                if self.done[b]:
                    nb_idx[b, lo: lo + gs] = lo
                    continue
                glp = lp[b, lo: lo + gs]
                if g > 0:
                    count = torch.bincount(nb_tokens[b, :lo], minlength=V).to(torch.float32)
                    glp = glp - self.lam * count
                glp = apply(glp, d_rows[b * K + lo: b * K + lo + gs], self.procs, self.bad_words)     # changed: + bad words
                sc = (glp + self.beam_scores[b, lo: lo + gs, None]).reshape(1, -1)
                val, idx = top_candidates(sc, 2 * gs)
                val, idx = val[0], idx[0]
                n = 0
                for rank in range(2 * gs):
                    flat = int(idx[rank]); beam, tok = lo + flat // V, flat % V
                    s = val[rank]
                    if tok == EOS:
                        if rank >= gs:
                            continue
                        self._add(b, self.tokens[b, beam, : self.t].tolist(), s.item(), cur_len)
                    else:
                        nb_scores[b, lo + n] = s; nb_tokens[b, lo + n] = tok; nb_idx[b, lo + n] = beam
                        n += 1
                    if n == gs:
                        break
                assert n == gs
                if self._is_done(b, val.max().item(), cur_len):                                      # changed: is_done
                    self.done[b] = True
        new_tokens = self.tokens.gather(1, nb_idx[:, :, None].expand(-1, -1, self.T)).clone()
        new_tokens[:, :, self.t] = nb_tokens
        self.tokens, self.beam_scores = new_tokens, nb_scores
        self.last_beam_idx, self.last_tokens = nb_idx, nb_tokens
        self.t += 1
        return nb_idx, nb_tokens, nb_scores


class ArgsBeamSampleState(_LengthPenalty, ProcessedBeamSampleState):
    """ProcessedBeamSampleState with length_penalty, early_stopping and bad words (the two marked lines)."""

    def __init__(self, B, K, V, max_new=18, N=1, temperature=1.0, top_k=7, top_p=0.0, seed=0, row_offset=0, prefix=None, processors=None,
                 length_penalty=1.0, early_stopping=False, bad_words_ids=None):
        super().__init__(B, K, V, max_new, N, temperature, top_k, top_p, seed, row_offset, prefix, processors)
        self._set_length_args(length_penalty, early_stopping)
        self.bad_words = check_bad_words(bad_words_ids, V)

    def step(self, logits, ngram_blocking_size=0, hist=None):
        S, K, V, N = self.B, self.K, self.V, self.N
        cur_len = self.t + self.P
        lg = logits.float()
        lp = lg - log_z(lg)
        if ngram_blocking_size > 0:
            for row, toks in enumerate(self.banned(hist, ngram_blocking_size)):
                for w in toks:
                    lp[row, w] = -float("inf")
        lp = apply(lp, self.decoder_inputs(), self.procs, self.bad_words)                          # changed: + bad words
        sc = lp + self.beam_scores.reshape(S * K, 1)
        val, idx = top_candidates(sc, NSEL)
        w = (val / self.temperature).reshape(S, K, NSEL)
        idx = idx.reshape(S, K, NSEL)
        kept = torch.tensor([[kept_count(w[s, k].numpy(), self.top_k, self.top_p) for k in range(K)] for s in range(S)])
        self.last_lists, self.last_draw = (w.clone(), idx.clone(), kept.clone()), []
        nb_scores = torch.zeros(S, K, dtype=torch.float32)
        nb_tokens = torch.zeros(S, K, dtype=torch.int64)
        nb_idx = torch.zeros(S, K, dtype=torch.int64)
        flat_all = (torch.arange(K)[:, None] * V + idx).reshape(S, K * NSEL)
        for s in range(S):
            if self.done[s]:
                self.last_draw.append(None)
                continue
            b, n = divmod(s, N)
            wv = w[s].reshape(-1).numpy()
            fl = flat_all[s].numpy()
            live = np.array([j < int(kept[s, k]) for k in range(K) for j in range(NSEL)])
            keys = np.full(K * NSEL, -np.inf)
            if live.any():
                u = uniforms(candidate_seed(self.seed, n), self.row_offset + b, self.t, fl[live])
                keys[live] = gumbel_keys(wv[live], u)
            draw = sorted(range(K * NSEL), key=lambda c: (-keys[c], c))[: 2 * K]
            draw.sort(key=lambda c: (-float(wv[c]), int(fl[c]), c))
            self.last_draw.append(draw)
            cnt = 0
            for rank, c in enumerate(draw):
                beam, tok = int(fl[c]) // V, int(fl[c]) % V
                v = float(wv[c])
                if tok == EOS:
                    if rank >= K:
                        continue
                    self._add(s, self.tokens[s, beam, : self.t].tolist(), v, cur_len)
                else:
                    nb_scores[s, cnt] = v; nb_tokens[s, cnt] = tok; nb_idx[s, cnt] = beam
                    cnt += 1
                if cnt == K:
                    break
            assert cnt == K
            if self._is_done(s, float(wv[draw[0]]), cur_len):                                         # changed: is_done
                self.done[s] = True
        new_tokens = self.tokens.gather(1, nb_idx[:, :, None].expand(-1, -1, self.T)).clone()
        new_tokens[:, :, self.t] = nb_tokens
        self.tokens, self.beam_scores = new_tokens, nb_scores
        self.last_beam_idx, self.last_tokens = nb_idx, nb_tokens
        self.t += 1
        return nb_idx, nb_tokens, nb_scores


def group_beam_state(sd, enc_cfg, dec_cfg, batch, num_beams, num_beam_groups=1, diversity_penalty=0.0, max_new=18, ngram_blocking_size=0,
                     prefix=None, processors=None, length_penalty=1.0, early_stopping=False, bad_words_ids=None):
    """oracle.processors.group_beam_state with the three arguments: the state before finalisation (``finalize`` /
    ``oracle.beam_nbest.finalize_nbest``)."""
    B, K = batch["enc_input_ids"].shape[0], num_beams
    enc_h, enc_m, hist = _encoded(sd, enc_cfg, batch, K)
    st = ArgsGroupBeamState(B, K, dec_cfg.vocab_size, max_new, num_beam_groups, diversity_penalty, prefix, processors, length_penalty,
                            early_stopping, bad_words_ids)
    start = st.prefix.repeat_interleave(K, 0)
    for t in range(max_new):
        h = R.decoder_hidden(sd, dec_cfg, torch.cat((start, st.tokens.reshape(B * K, -1)[:, :t]), 1), None, enc_h, enc_m)
        st.step(R.lm_logits(sd, h[:, -1]), ngram_blocking_size, hist)
        if bool(st.done.all()):
            break
    return st


def beam_sample(sd, enc_cfg, dec_cfg, batch, num_beams, N=1, temperature=0.7, top_k=7, top_p=0.0, seed=0, row_offset=0, max_new=18,
                ngram_blocking_size=0, prefix=None, processors=None, length_penalty=1.0, early_stopping=False, bad_words_ids=None):
    """oracle.processors.beam_sample with the three arguments: (sequences, scores)."""
    B, K = batch["enc_input_ids"].shape[0], num_beams
    enc_h, enc_m, hist = _encoded(sd, enc_cfg, batch, N * K)
    st = ArgsBeamSampleState(B, K, dec_cfg.vocab_size, max_new, N, temperature, top_k, top_p, seed, row_offset, prefix, processors,
                             length_penalty, early_stopping, bad_words_ids)
    start = st.prefix.repeat_interleave(K, 0)
    for t in range(max_new):
        h = R.decoder_hidden(sd, dec_cfg, torch.cat((start, st.tokens.reshape(B * N * K, -1)[:, :t]), 1), None, enc_h, enc_m)
        st.step(R.lm_logits(sd, h[:, -1]), ngram_blocking_size, hist)
        if bool(st.done.all()):
            break
    return st.finalize()


def generate_greedy_or_sample(sd, enc_cfg, dec_cfg, batch, temperature=1.0, top_k=1, top_p=0.0, ngram_blocking_size=0, max_new=18,
                              generator=None, processors=None, bad_words_ids=None):
    """oracle.processors.generate_greedy_or_sample with the bad words, applied with the processors after the temperature."""
    procs = _checked(processors)
    bad = check_bad_words(bad_words_ids, dec_cfg.vocab_size)
    ids, seg, att = batch["enc_input_ids"], batch["enc_segments"], batch["enc_att_mask"]
    seq_t, seq_v = R.encoder(sd, enc_cfg, ids, batch["enc_image_feat"], batch["enc_image_loc"], seg, att, batch["enc_image_mask"])
    enc_h, enc_m = R.vlfusion(sd, seq_t, seq_v, att, batch["enc_image_mask"])
    dec_ids = batch["dec_input_ids"].clone()
    hist = (ids * (seg == 0).long()).tolist()
    out = []
    for _ in range(max_new):
        _, logits = R.decoder_forward(sd, dec_cfg, dec_ids, None, enc_h, enc_m)
        step = logits[:, -1, :] / temperature
        step = apply(step, [LP.decoder_ids(r) for r in dec_ids.tolist()], procs, bad)                  # changed: + bad words
        if ngram_blocking_size > 0:
            for r in range(step.shape[0]):
                banned = R.ngram_banned_tokens(hist[r], dec_ids[r].tolist(), ngram_blocking_size)
                step[r, banned] = -float("inf")
        step = R.top_k_top_p_filter(step, top_k, top_p)
        prob = torch.softmax(step, dim=-1)
        nxt = prob.argmax(-1, keepdim=True) if top_k == 1 else torch.multinomial(prob, 1, generator=generator)
        dec_ids = torch.cat((dec_ids, nxt), dim=-1)
        out.append(nxt)
    seq = torch.cat(out, 1)
    mask = torch.zeros_like(seq)
    for e in (seq == EOS).nonzero(as_tuple=False):
        mask[e[0], e[1] + 1:] = 1
    return seq.masked_fill(mask.bool(), PAD)


def completes_bad_word(d, seq, bad_words_ids):
    """True when some listed sequence (not [SEP] alone) ends at a position of ``seq`` (the generated tokens up to their first [SEP],
    exclusive) appended to decoder input ``d`` - i.e. the output completed a banned sequence."""
    full = list(d)
    for w in seq:
        if int(w) in bad_words_banned(full, bad_words_ids):
            return True
        full.append(int(w))
    return False
