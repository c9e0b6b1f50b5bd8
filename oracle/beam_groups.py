"""TEST INFRASTRUCTURE ONLY - diverse (group) beam search: beam groups with a Hamming diversity penalty (plain PyTorch / Python, CPU).

Restates ``transformers==4.16.2`` ``GenerationMixin.group_beam_search`` + ``BeamSearchScorer(num_beam_groups=G)`` +
``HammingDiversityLogitsProcessor`` (``num_beam_groups`` / ``diversity_penalty``), the published algorithm of Vijayakumar et al.,
"Diverse Beam Search: Decoding Diverse Solutions from Neural Sequence Models" (AAAI 2018), on top of the arithmetic of
oracle/beam.py and oracle/beam_ngram.py, which are unchanged.  Parity is UNPINNED against a reference implementation: the
reference has no beam search and transformers 4.16.2 is not available to run against; the CUDA beam step must match THIS file
bit-exactly on indices when both are fed the same fp32 logits.

Setup: K beams, G groups with G | K, group size gs = K / G, penalty lambda >= 0 (fp32).
  * init: beam k of an image starts with score 0 if k % gs == 0, else -1e9 (HF ``beam_scores[:, ::num_sub_beams] = 0``)
  * one decoder pass over all K rows per step; logZ per row as in oracle/beam.py, over the full unbanned row
  * within a step the groups g = 0 .. G-1 run in order.  Candidate (beam k of group g, token w) =
      fp32(fp32(fp32(x - logZ) - fp32(lambda * c_w)) + beam_score_k)
    with c_w = how many new beams of groups 0..g-1 of the same image took token w at this step (an EOS that closed a hypothesis
    is not appended to a beam and does not count).  c_w = 0 gives oracle/beam.py's fp32(fp32(x - logZ) + beam_score) exactly.
    A token banned by n-gram blocking (oracle/beam_ngram.py) is -inf before the penalty and stays -inf.
  * per group: the top 2*gs of its gs*V candidates by (score desc, local flat index (k - g*gs)*V + w asc), then
    ``BeamSearchScorer.process`` with group_size = gs: EOS is added to the hypotheses only at rank < gs, the group gets gs new
    beams, parents stay inside the group
  * one hypothesis heap of capacity K per image, shared by all groups; ``done`` is per image, tested at the START of every group's
    process (once group g finishes an image, groups g+1.. of the same step are padded: score 0, token PAD, parent = the group's
    first beam) and updated after every group with ``is_done(max of that group's 2*gs candidate scores, cur_len)``
  * finalize: unchanged (``BeamSearchScorer.finalize`` over all K beams of an undone image; N-best pop order of oracle/beam_nbest.py)
With G = 1 every step gives exactly the ids and scores of ``BlockedBeamState`` (any lambda: group 0 is never penalised).

Decoder prefix: ``prefix`` int64 [B, P] (None = one [CLS] per row) with the semantics of the prefix beam state of
tests/test_decoder_prefix.py: a [SEP] in the prefix is read as [PAD], n-gram keys may reach into it, and hypothesis lengths are
P + t.  ``P`` is exposed so that ``oracle.beam_nbest.finalize_nbest`` works on this state unchanged.
"""
from __future__ import annotations

import math

import torch

from . import restatement as R
from .beam import EOS, PAD, log_z, top_candidates
from .beam_nbest import finalize_nbest
from .beam_ngram import BlockedBeamState, question_history


def decoder_input(prefix, B):
    """int64 [B, P] decoder input of a caller's prefix with [SEP] read as [PAD]; None -> one [CLS] per row."""
    if prefix is None:
        return torch.full((B, 1), R.CLS, dtype=torch.int64)
    p = prefix.to(torch.int64).clone()
    return p.masked_fill(p == EOS, PAD)


def check_group_args(K, num_beam_groups, diversity_penalty):
    G, lam = int(num_beam_groups), float(diversity_penalty)
    if G < 1 or K % G != 0:
        raise ValueError(f"num_beam_groups must divide num_beams ({K}), got {G}")
    if not (math.isfinite(lam) and lam >= 0.0):
        raise ValueError(f"diversity_penalty must be finite and >= 0, got {diversity_penalty}")
    return G, lam


class GroupBeamState(BlockedBeamState):
    """Beam state of HF 4.16.2 ``group_beam_search`` (contract above)."""

    def __init__(self, B, K, V, max_new=18, num_beam_groups=1, diversity_penalty=0.0, prefix=None):
        G, lam = check_group_args(K, num_beam_groups, diversity_penalty)
        super().__init__(B, K, V, max_new)
        self.G, self.gs = G, K // G
        self.lam = torch.tensor(lam, dtype=torch.float32)                 # the penalty is an fp32 operand
        self.beam_scores.fill_(-1e9)
        self.beam_scores[:, ::self.gs] = 0.0
        self.prefix = decoder_input(prefix, B)
        self.P = self.prefix.shape[1]

    def banned(self, hist, n):
        return [R.ngram_banned_tokens(hist[b], self.prefix[b].tolist() + self.tokens[b, k, : self.t].tolist(), n) if n > 0 else []
                for b in range(self.B) for k in range(self.K)]

    def step(self, logits, ngram_blocking_size=0, hist=None):
        B, K, V, G, gs = self.B, self.K, self.V, self.G, self.gs
        cur_len = self.t + self.P
        lg = logits.float()
        lp = (lg - log_z(lg)).reshape(B, K, V)                             # fp32(x - logZ)
        if ngram_blocking_size > 0:
            for row, toks in enumerate(self.banned(hist, ngram_blocking_size)):
                b, k = divmod(row, K)
                for w in toks:
                    lp[b, k, w] = -float("inf")
        nb_scores = torch.zeros(B, K, dtype=torch.float32)
        nb_tokens = torch.zeros(B, K, dtype=torch.int64)
        nb_idx = torch.zeros(B, K, dtype=torch.int64)
        for b in range(B):
            for g in range(G):
                lo = g * gs
                if self.done[b]:
                    nb_idx[b, lo: lo + gs] = lo                            # padded: score 0, token PAD
                    continue
                glp = lp[b, lo: lo + gs]
                if g > 0:
                    count = torch.bincount(nb_tokens[b, :lo], minlength=V).to(torch.float32)
                    glp = glp - self.lam * count                           # fp32(lp - fp32(lambda * c)); -inf stays -inf
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

    def finalize(self):
        return finalize_nbest(self, 1)


def group_beam_state(sd, enc_cfg, dec_cfg, batch, num_beams, num_beam_groups=1, diversity_penalty=0.0, max_new=18,
                     ngram_blocking_size=0, prefix=None):
    """Runs group beam search over the restated reference modules (no KV cache, whole decoder input every step) and returns the
    state before finalisation (``finalize`` / ``oracle.beam_nbest.finalize_nbest``)."""
    ids, seg, att = batch["enc_input_ids"], batch["enc_segments"], batch["enc_att_mask"]
    B, K = ids.shape[0], num_beams
    seq_t, seq_v = R.encoder(sd, enc_cfg, ids, batch["enc_image_feat"], batch["enc_image_loc"], seg, att, batch["enc_image_mask"])
    enc_h, enc_m = R.vlfusion(sd, seq_t, seq_v, att, batch["enc_image_mask"])
    enc_h, enc_m = enc_h.repeat_interleave(K, 0), enc_m.repeat_interleave(K, 0)
    hist = question_history(ids, seg)
    st = GroupBeamState(B, K, dec_cfg.vocab_size, max_new, num_beam_groups, diversity_penalty, prefix)
    start = st.prefix.repeat_interleave(K, 0)
    for t in range(max_new):
        h = R.decoder_hidden(sd, dec_cfg, torch.cat((start, st.tokens.reshape(B * K, -1)[:, :t]), 1), None, enc_h, enc_m)
        st.step(R.lm_logits(sd, h[:, -1]), ngram_blocking_size, hist)
        if bool(st.done.all()):
            break
    return st
