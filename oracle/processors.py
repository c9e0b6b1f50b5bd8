"""TEST INFRASTRUCTURE ONLY - HF logits processors on per-row decoder inputs (plain PyTorch / Python, CPU).

Restates the three ``transformers`` processors that stop degenerate output, as ``gstvd_generate`` applies them (include/gstvd.h):
``RepetitionPenaltyLogitsProcessor``, ``NoRepeatNGramLogitsProcessor`` and ``MinLengthLogitsProcessor``.  For 2-D scores their code is
the same in 4.16.2 (the reference's pin) and in the installed 5.x; ``oracle/gen_golden_processors.py`` pins this file on HF's own
classes and writes tests/golden/logits_processors.npz.

Contract, for scores s [rows, V] fp32 and per-row decoder inputs d (HF input_ids: the image's decoder prefix with [SEP] read as [PAD],
[CLS] when there is none, then the row's own generated tokens), cur_len = len(d):
  1. repetition_penalty p (1 = off): every distinct id of d gets s < 0 ? fp32(s * p) : fp32(s / p) - once per id however often it
     occurs (HF's gather / scatter);
  2. no_repeat_ngram_size n (0 = off), only when cur_len + 1 >= n: wherever the last n-1 ids of d occur earlier in d, the id that
     follows them there gets -inf.  No special id is exempt: n = 1 bans every id of d;
  3. min_length m (0 = off): [SEP] (102) gets -inf while cur_len < m (decoder-input length, prefix included, as in 4.16.2).
-inf stays -inf.  The processors run in this order (HF ``_get_logits_processor``); the result does not depend on it, since the two
later ones only write -inf.  In beam groups HF 4.16.2 runs ``HammingDiversityLogitsProcessor`` before all three (that processor left
the library with group beam search, so the installed 5.x cannot be run against; ``ProcessedGroupBeamState`` below applies the order).

The decode oracles with the processors are at the end of this file: ``generate_greedy_or_sample`` (sampling), ``ProcessedGroupBeamState``
/ ``group_beam_state`` (beam search, with or without groups and a decoder prefix) and ``ProcessedBeamSampleState`` / ``beam_sample``.
"""
from __future__ import annotations

import math

import numpy as np
import torch

EOS, PAD = 102, 0


def decoder_ids(ids):
    """A decoder input as a list with [SEP] read as [PAD] (the key the question-history blocking uses as well)."""
    return [PAD if int(w) == EOS else int(w) for w in ids]


def check_args(repetition_penalty=1.0, no_repeat_ngram_size=0, min_length=0):
    if not (math.isfinite(repetition_penalty) and repetition_penalty > 0.0):
        raise ValueError(f"repetition_penalty must be finite and > 0, got {repetition_penalty}")
    if int(no_repeat_ngram_size) < 0 or int(min_length) < 0:
        raise ValueError("no_repeat_ngram_size and min_length must be >= 0")


def active(repetition_penalty=1.0, no_repeat_ngram_size=0, min_length=0):
    return repetition_penalty != 1.0 or no_repeat_ngram_size > 0 or min_length > 0


def no_repeat_ngram_banned(d, n):
    """The ids NoRepeatNGramLogitsProcessor bans for one row with decoder input d (a list)."""
    L = len(d)
    if n <= 0 or L + 1 < n:
        return []
    key = tuple(d[L - n + 1:]) if n > 1 else ()
    return [d[i + n - 1] for i in range(L - n + 1) if tuple(d[i:i + n - 1]) == key]


def repetition_penalize(s, ids, p):
    """fp32 s of the ids (1-D tensor or list) penalised once: s < 0 ? s * p : s / p."""
    p = torch.tensor(p, dtype=torch.float32)
    return torch.where(s < 0, s * p, s / p)


def apply(scores, d_rows, repetition_penalty=1.0, no_repeat_ngram_size=0, min_length=0):
    """The three processors on scores [rows, V] fp32 (a new tensor); d_rows: per-row decoder inputs (lists of ids)."""
    out = scores.float().clone()
    if not active(repetition_penalty, no_repeat_ngram_size, min_length):
        return out
    for r, d in enumerate(d_rows):
        d = [int(w) for w in d]
        if repetition_penalty != 1.0 and d:
            ids = torch.tensor(sorted(set(d)), dtype=torch.int64)
            out[r, ids] = repetition_penalize(out[r, ids], ids, repetition_penalty)
        if no_repeat_ngram_size > 0:
            banned = no_repeat_ngram_banned(d, no_repeat_ngram_size)
            if banned:
                out[r, torch.tensor(banned, dtype=torch.int64)] = -float("inf")
        if len(d) < min_length:
            out[r, EOS] = -float("inf")
    return out


def has_repeated_ngram(d, n):
    """True when some n-gram occurs twice in d."""
    grams = [tuple(d[i:i + n]) for i in range(len(d) - n + 1)]
    return len(grams) != len(set(grams))


# ---- the decode oracles with the processors ------------------------------------------------------------------------------
# The oracles of oracle/restatement.py, oracle/beam_groups.py and oracle/beam_sample.py, unchanged, with the processors added at the
# point gstvd_generate applies them.  Each step below is its base class's step with one added line (marked); with the processors off
# it computes exactly what the base class computes (tests/test_logits_processors.py checks it).
from . import restatement as R  # noqa: E402
from .beam import log_z, top_candidates  # noqa: E402
from .beam_groups import GroupBeamState  # noqa: E402
from .beam_ngram import question_history  # noqa: E402
from .beam_sample import BeamSampleState, candidate_seed, gumbel_keys, kept_count, uniforms, NSEL  # noqa: E402


def _checked(processors):
    p = dict(dict(repetition_penalty=1.0, no_repeat_ngram_size=0, min_length=0), **(processors or {}))
    check_args(**p)
    return p


class ProcessedGroupBeamState(GroupBeamState):
    """HF beam search (num_beam_groups = 1, which is plain beam search with a decoder prefix) and group beam search with the logits
    processors: they act on fp32(x - logZ) with the beam's decoder input, after the Hamming term (HF 4.16.2's processor order), before
    the beam score is added."""

    def __init__(self, B, K, V, max_new=18, num_beam_groups=1, diversity_penalty=0.0, prefix=None, processors=None):
        super().__init__(B, K, V, max_new, num_beam_groups, diversity_penalty, prefix)
        self.procs = _checked(processors)

    def decoder_inputs(self):
        return [decoder_ids(self.prefix[b].tolist() + self.tokens[b, k, : self.t].tolist()) for b in range(self.B) for k in range(self.K)]

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
                glp = apply(glp, d_rows[b * K + lo: b * K + lo + gs], **self.procs)                 # added: the processors
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
                if len(self.hyps[b]) >= K and self.worst[b] >= float(val.max().item()) / float(cur_len):
                    self.done[b] = True
        new_tokens = self.tokens.gather(1, nb_idx[:, :, None].expand(-1, -1, self.T)).clone()
        new_tokens[:, :, self.t] = nb_tokens
        self.tokens, self.beam_scores = new_tokens, nb_scores
        self.last_beam_idx, self.last_tokens = nb_idx, nb_tokens
        self.t += 1
        return nb_idx, nb_tokens, nb_scores


class ProcessedBeamSampleState(BeamSampleState):
    """HF beam sampling with the logits processors: on fp32(x - logZ) with the beam's decoder input, next to the n-gram bans, before the
    beam score is added and the warpers act."""

    def __init__(self, B, K, V, max_new=18, N=1, temperature=1.0, top_k=7, top_p=0.0, seed=0, row_offset=0, prefix=None, processors=None):
        super().__init__(B, K, V, max_new, N, temperature, top_k, top_p, seed, row_offset, prefix)
        self.procs = _checked(processors)

    def decoder_inputs(self):
        return [decoder_ids(self.prefix[s].tolist() + self.tokens[s, k, : self.t].tolist()) for s in range(self.B) for k in range(self.K)]

    def step(self, logits, ngram_blocking_size=0, hist=None):
        S, K, V, N = self.B, self.K, self.V, self.N
        cur_len = self.t + self.P
        lg = logits.float()
        lp = lg - log_z(lg)
        if ngram_blocking_size > 0:
            for row, toks in enumerate(self.banned(hist, ngram_blocking_size)):
                for w in toks:
                    lp[row, w] = -float("inf")
        lp = apply(lp, self.decoder_inputs(), **self.procs)                                          # added: the processors
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
            if len(self.hyps[s]) >= K and self.worst[s] >= float(wv[draw[0]]) / float(cur_len):
                self.done[s] = True
        new_tokens = self.tokens.gather(1, nb_idx[:, :, None].expand(-1, -1, self.T)).clone()
        new_tokens[:, :, self.t] = nb_tokens
        self.tokens, self.beam_scores = new_tokens, nb_scores
        self.last_beam_idx, self.last_tokens = nb_idx, nb_tokens
        self.t += 1
        return nb_idx, nb_tokens, nb_scores


def _encoded(sd, enc_cfg, batch, rows_per_image):
    ids, seg, att = batch["enc_input_ids"], batch["enc_segments"], batch["enc_att_mask"]
    seq_t, seq_v = R.encoder(sd, enc_cfg, ids, batch["enc_image_feat"], batch["enc_image_loc"], seg, att, batch["enc_image_mask"])
    enc_h, enc_m = R.vlfusion(sd, seq_t, seq_v, att, batch["enc_image_mask"])
    return enc_h.repeat_interleave(rows_per_image, 0), enc_m.repeat_interleave(rows_per_image, 0), question_history(ids, seg)


def group_beam_state(sd, enc_cfg, dec_cfg, batch, num_beams, num_beam_groups=1, diversity_penalty=0.0, max_new=18, ngram_blocking_size=0,
                     prefix=None, processors=None):
    """oracle.beam_groups.group_beam_state with the logits processors: the state before finalisation."""
    B, K = batch["enc_input_ids"].shape[0], num_beams
    enc_h, enc_m, hist = _encoded(sd, enc_cfg, batch, K)
    st = ProcessedGroupBeamState(B, K, dec_cfg.vocab_size, max_new, num_beam_groups, diversity_penalty, prefix, processors)
    start = st.prefix.repeat_interleave(K, 0)
    for t in range(max_new):
        h = R.decoder_hidden(sd, dec_cfg, torch.cat((start, st.tokens.reshape(B * K, -1)[:, :t]), 1), None, enc_h, enc_m)
        st.step(R.lm_logits(sd, h[:, -1]), ngram_blocking_size, hist)
        if bool(st.done.all()):
            break
    return st


def beam_sample(sd, enc_cfg, dec_cfg, batch, num_beams, N=1, temperature=0.7, top_k=7, top_p=0.0, seed=0, row_offset=0, max_new=18,
                ngram_blocking_size=0, prefix=None, processors=None):
    """oracle.beam_sample.beam_sample with the logits processors: (sequences, scores)."""
    B, K = batch["enc_input_ids"].shape[0], num_beams
    enc_h, enc_m, hist = _encoded(sd, enc_cfg, batch, N * K)
    st = ProcessedBeamSampleState(B, K, dec_cfg.vocab_size, max_new, N, temperature, top_k, top_p, seed, row_offset, prefix, processors)
    start = st.prefix.repeat_interleave(K, 0)
    for t in range(max_new):
        h = R.decoder_hidden(sd, dec_cfg, torch.cat((start, st.tokens.reshape(B * N * K, -1)[:, :t]), 1), None, enc_h, enc_m)
        st.step(R.lm_logits(sd, h[:, -1]), ngram_blocking_size, hist)
        if bool(st.done.all()):
            break
    return st.finalize()


def generate_greedy_or_sample(sd, enc_cfg, dec_cfg, batch, temperature=1.0, top_k=1, top_p=0.0, ngram_blocking_size=0, max_new=18,
                              generator=None, processors=None):
    """oracle.restatement.generate_greedy_or_sample with the logits processors, applied after the temperature (the order of the
    reference's loop) on each row's dec_ids with [SEP] read as [PAD]."""
    procs = _checked(processors)
    ids, seg, att = batch["enc_input_ids"], batch["enc_segments"], batch["enc_att_mask"]
    seq_t, seq_v = R.encoder(sd, enc_cfg, ids, batch["enc_image_feat"], batch["enc_image_loc"], seg, att, batch["enc_image_mask"])
    enc_h, enc_m = R.vlfusion(sd, seq_t, seq_v, att, batch["enc_image_mask"])
    dec_ids = batch["dec_input_ids"].clone()
    hist = (ids * (seg == 0).long()).tolist()
    out = []
    for _ in range(max_new):
        _, logits = R.decoder_forward(sd, dec_cfg, dec_ids, None, enc_h, enc_m)
        step = logits[:, -1, :] / temperature
        step = apply(step, [decoder_ids(r) for r in dec_ids.tolist()], **procs)                        # added: the processors
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
