"""TEST INFRASTRUCTURE ONLY - beam sampling: ``num_beams`` > 1 with ``do_sample`` (plain PyTorch / Python, CPU).

Restates ``transformers==4.16.2`` ``GenerationMixin.generate`` -> ``beam_sample`` + ``BeamSearchScorer`` (``length_penalty = 1``,
``early_stopping = False``) with its logits warpers (``TemperatureLogitsWarper``, ``TopKLogitsWarper`` / ``TopPLogitsWarper`` with
``min_tokens_to_keep = 2``), on top of the arithmetic of oracle/beam.py and oracle/beam_ngram.py, which are unchanged.  Parity is
UNPINNED against a reference implementation: the reference has no beam search and transformers 4.16.2 is not available to run
against; the CUDA beam-sample step must match THIS file bit-exactly on indices when both are fed the same fp32 logits.

Setup: K >= 2 beams per search, N independent searches per image (HF ``num_return_sequences = N`` with ``beam_sample`` expands the
input N times, so every output is the best hypothesis of its own search), temperature T > 0, top_k in 1..16, top_p in [0, 1] (0 = off),
seed, row_offset.  Search n of image b is search s = b*N + n; its beam k is decode row s*K + k.  Per search and step t:
  1. init: all K beams start at score 0 (``beam_sample`` does not set beams 1..K-1 to -1e9 the way ``beam_search`` does).
  2. s = fp32(fp32(x - logZ) + beam_score) per (beam k, token w), logZ as in oracle/beam.py over the full row; n-gram-banned tokens
     (oracle/beam_ngram.py; keys may reach into the decoder prefix) are -inf before the beam score is added.
  3. warpers per row, in HF order and AFTER the beam score is added (4.16.2 behaviour: the temperature compounds through the beam
     scores, since every new beam score is a warped value that the next step divides by T again):
       w = fp32(s / T);
       each row keeps its 16 best by (s desc, token asc) - the candidate list of the CUDA row selection; w is monotone in s, so the
       list is also ordered by w;
       top-k: keep w >= the k'-th listed w, k' = max(top_k, 2) (ties at the threshold as far as the 16 reach; -inf never kept);
       top-p (> 0): inside the kept prefix, p_r = fp32 exp(w_r - w_0), Z = their fp32 sum in order, and rank r >= 2 is dropped (with
       every later rank) when the fp32 running sum of fp32(p_i / Z), i < r, exceeds top_p.
  4. draw 2K entries without replacement from softmax(w) over the K*V entries (HF ``torch.multinomial(probs, 2K)``) by Gumbel-top-2K:
     key = fp64(w) - log(-log(u)) in fp64 for the kept entries, -inf for the others; the 2K largest keys (ties: list position
     k*16 + j asc) are drawn.  u = ((h >> 11) + 0.5) * 2^-53 with
       h = splitmix64(splitmix64(sd ^ splitmix64(((row_offset + b) << 20) ^ t)) ^ (k*V + w)),  sd = candidate_seed(seed, n).
     Gumbel-top-k has the law of sequential sampling without replacement, works in the log domain and never underflows; HF raises
     when fewer than 2K probabilities are non-zero in fp32, this draw still draws.
  5. the drawn entries sorted by (w desc, k*V + w asc), then ``BeamSearchScorer.process`` as in oracle/beam.py: [SEP] becomes a
     hypothesis only at rank < K, with score (warped sum) / (P + t); the other tokens fill the K new beams; ``is_done`` with the best
     drawn w.  A search that is done is padded (score 0, token PAD, parent 0).
  6. finalize: oracle/beam_nbest.py with one return sequence per search; output row b*N + n is search n's best hypothesis.
"""
from __future__ import annotations

import math

import numpy as np
import torch

from . import restatement as R
from .beam import EOS, PAD, log_z, top_candidates
from .beam_groups import decoder_input
from .beam_nbest import finalize_nbest
from .beam_ngram import BlockedBeamState, question_history

NSEL = 16                                           # per-row candidate list of the CUDA row selection (kSelMax)
M64 = 0xFFFFFFFFFFFFFFFF


def splitmix64(x):
    """splitmix64 on uint64 numpy arrays (wrapping arithmetic)."""
    x = np.asarray(x, dtype=np.uint64) + np.uint64(0x9E3779B97F4A7C15)
    x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return x ^ (x >> np.uint64(31))


def candidate_seed(seed, n):
    """Mirror of candidate_seed in csrc/select.cu (also models/visual_dialog_model.candidate_seed)."""
    seed = int(seed) & M64
    if int(n) == 0:
        return seed
    return int(splitmix64(np.array([seed ^ int(splitmix64(np.array([(int(n) * 0xD1B54A32D192ED03) & M64]))[0])], dtype=np.uint64))[0])


def uniforms(sd, grow, t, flat):
    """u in (0, 1) for the flat indices ``flat`` (k*V + w) of one search and step: the counter-based RNG of the draw."""
    inner = int(splitmix64(np.array([(((int(grow) << 20) & M64) ^ int(t))], dtype=np.uint64))[0])
    base = int(splitmix64(np.array([int(sd) ^ inner], dtype=np.uint64))[0])
    h = splitmix64(np.uint64(base) ^ np.asarray(flat, dtype=np.uint64).reshape(-1))
    return ((h >> np.uint64(11)).astype(np.float64) + 0.5) * 2.0 ** -53


def gumbel_keys(w, u):
    """fp64(w) - log(-log(u)), w fp32 values."""
    return np.asarray(w, dtype=np.float32).astype(np.float64) - np.log(-np.log(u))


def kept_count(w, top_k, top_p):
    """Warpers on one row's list ``w`` (fp32, 16 entries, descending): the number of leading entries kept."""
    w = np.asarray(w, dtype=np.float32)
    thr = w[max(int(top_k), 2) - 1]
    kept = 0
    while kept < len(w) and w[kept] >= thr and w[kept] > -np.inf:
        kept += 1
    if top_p > 0.0 and kept > 2:
        p = np.exp((w[:kept] - w[0]).astype(np.float32)).astype(np.float32)
        tot = np.float32(0.0)
        for x in p:
            tot = np.float32(tot + x)
        cum = np.float32(0.0)
        for r in range(kept):
            if r >= 2 and cum > np.float32(top_p):
                kept = r
                break
            cum = np.float32(cum + np.float32(p[r] / tot))
    return kept


def check_sample_args(K, N, temperature, top_k, top_p):
    if K < 2 or 2 * K > NSEL:
        raise ValueError(f"beam sampling needs 2 <= num_beams <= {NSEL // 2}, got {K}")
    if N < 1:
        raise ValueError(f"num_return_sequences must be >= 1, got {N}")
    if not (math.isfinite(temperature) and temperature > 0.0):
        raise ValueError(f"temperature must be finite and > 0, got {temperature}")
    if not 0.0 <= top_p <= 1.0:
        raise ValueError(f"top_p must be in [0, 1], got {top_p}")
    if not 1 <= top_k <= NSEL:
        raise ValueError(f"top_k must be in 1..{NSEL}, got {top_k}")


class BeamSampleState(BlockedBeamState):
    """B*N searches of K beams (contract above).  ``B`` counts images; ``self.B`` the searches."""

    def __init__(self, B, K, V, max_new=18, N=1, temperature=1.0, top_k=7, top_p=0.0, seed=0, row_offset=0, prefix=None):
        check_sample_args(K, N, temperature, top_k, top_p)
        super().__init__(B * N, K, V, max_new)
        self.images, self.N = B, N
        self.temperature = torch.tensor(temperature, dtype=torch.float32)
        self.top_k, self.top_p = int(top_k), float(top_p)
        self.seed, self.row_offset = int(seed) & M64, int(row_offset)
        self.beam_scores.zero_()
        self.prefix = decoder_input(prefix, B).repeat_interleave(N, 0)
        self.P = self.prefix.shape[1]
        self.last_lists = None                      # per step: (w [S, K, 16], idx [S, K, 16], kept [S, K]) for property tests
        self.last_draw = None                       # per search: drawn list positions k*16 + j in the order given to the scorer

    def banned(self, hist, n):
        return [R.ngram_banned_tokens(hist[s // self.N], self.prefix[s].tolist() + self.tokens[s, k, : self.t].tolist(), n) if n > 0 else []
                for s in range(self.B) for k in range(self.K)]

    def step(self, logits, ngram_blocking_size=0, hist=None):
        S, K, V, N = self.B, self.K, self.V, self.N
        cur_len = self.t + self.P
        lg = logits.float()
        lp = lg - log_z(lg)                                               # fp32(x - logZ), [S*K, V]
        if ngram_blocking_size > 0:
            for row, toks in enumerate(self.banned(hist, ngram_blocking_size)):
                for w in toks:
                    lp[row, w] = -float("inf")
        sc = lp + self.beam_scores.reshape(S * K, 1)
        val, idx = top_candidates(sc, NSEL)                               # per row, (s desc, token asc)
        w = (val / self.temperature).reshape(S, K, NSEL)                  # fp32(s / T)
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
                continue                                                  # padded: score 0, token PAD, parent 0
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

    def finalize(self):
        """(sequences [B*N, T], scores [B*N] fp64): row b*N + n is the best hypothesis of search n of image b."""
        return finalize_nbest(self, 1)


def beam_sample(sd, enc_cfg, dec_cfg, batch, num_beams, N=1, temperature=0.7, top_k=7, top_p=0.0, seed=0, row_offset=0, max_new=18,
                ngram_blocking_size=0, prefix=None):
    """Beam sampling over the restated reference modules (no KV cache, whole decoder input every step): (sequences, scores)."""
    ids, seg, att = batch["enc_input_ids"], batch["enc_segments"], batch["enc_att_mask"]
    B, K = ids.shape[0], num_beams
    seq_t, seq_v = R.encoder(sd, enc_cfg, ids, batch["enc_image_feat"], batch["enc_image_loc"], seg, att, batch["enc_image_mask"])
    enc_h, enc_m = R.vlfusion(sd, seq_t, seq_v, att, batch["enc_image_mask"])
    enc_h, enc_m = enc_h.repeat_interleave(N * K, 0), enc_m.repeat_interleave(N * K, 0)
    hist = question_history(ids, seg)
    st = BeamSampleState(B, K, dec_cfg.vocab_size, max_new, N, temperature, top_k, top_p, seed, row_offset, prefix)
    start = st.prefix.repeat_interleave(K, 0)
    for t in range(max_new):
        h = R.decoder_hidden(sd, dec_cfg, torch.cat((start, st.tokens.reshape(B * N * K, -1)[:, :t]), 1), None, enc_h, enc_m)
        st.step(R.lm_logits(sd, h[:, -1]), ngram_blocking_size, hist)
        if bool(st.done.all()):
            break
    return st.finalize()
