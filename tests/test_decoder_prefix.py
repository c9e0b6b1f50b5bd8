"""Decoding from a caller-supplied decoder prefix (dec_input_ids [B, P]; include/gstvd.h gstvd_generate, its prefix / P arguments).

The beam contract with a prefix is defined here (``PrefixBeamState``, ``prefix_beam_search``) on top of oracle/beam.py and
oracle/beam_ngram.py, which define it for the [CLS] start.
CPU: that oracle reduces to oracle/beam.py / oracle/beam_ngram.py for the [CLS] start, never selects a banned (beam, token) pair when
the n-gram key reaches into the prefix, and the restatement continues its own greedy output from a prefix of it.
GPU: greedy ids identical to the restatement in fp32 (tiny and full size, P up to 25 = 42 cached positions), beam ids and scores
identical to the prefix oracle in fp32 on every call path, the bf16 product path agrees across call paths and an explicit [CLS]
prefix (P = 1) matches the implicit [CLS] start, and every rejected argument raises.
"""
import copy
import ctypes

import pytest
import torch

from helpers import R, history_batch
from oracle import beam as OB
from oracle import beam_ngram as BN

A4 = {"tiny": (500, 501, 502, 503), "full": (2000, 2001, 2002, 2003)}   # a question 4-gram spliced into every history
_GREEDY = dict(temperature=1.0, top_k=1, top_p=0.0)


def _with_bias(sd, add):
    """sd with the LM-head bias of the tokens in ``add`` raised (both names of the shared tensor)."""
    sd = dict(sd)
    bias = sd["decoder.decoder.lm_head.bias"].clone()
    for tok, v in add.items():
        bias[tok] += v
    sd["decoder.decoder.lm_head.bias"] = bias
    sd["decoder.decoder.lm_head.decoder.bias"] = bias
    return sd


def _with_question(b, toks):
    """Splices ``toks`` + [SEP] into every row's history as a question (segment 0)."""
    ids, seg = b["enc_input_ids"], b["enc_segments"]
    utt = torch.tensor(list(toks) + [R.EOS]).repeat(ids.shape[0], 1)
    R.splice(ids, seg, (ids != 0).sum(-1), utt, None, set())
    b["enc_att_mask"] = (ids != 0).float()
    return b


def _prefixes(B, P, vocab, seed=0):
    """[B, P] prefixes: row 0 starts with [CLS] and holds a [SEP], row 1 does not start with [CLS], row 2 holds [PAD]s."""
    g = torch.Generator().manual_seed(seed + P)
    p = torch.randint(1000 if vocab > 2000 else 200, vocab, (B, P), generator=g)
    p[:, 0] = R.CLS
    if B > 1:
        p[1, 0] = int(p[1, -1])
    if P > 2:
        p[0, P // 2] = R.EOS
        if B > 2:
            p[2, 1:P // 2] = R.PAD
    return p


def _greedy_ref(sd, enc_cfg, dec_cfg, b, prefix, n=0, max_new=18):
    bb = dict(b)
    bb["dec_input_ids"] = prefix
    with torch.no_grad():
        return R.generate_greedy_or_sample(sd, enc_cfg, dec_cfg, bb, 1.0, 1, 0.0, n, max_new=max_new)


# ---- beam oracle with a decoder prefix (test infrastructure, CPU) -----------------------------------------------------
def decoder_input(prefix, B):
    """The decoder input a caller's prefix stands for: int64 [B, P] with [SEP] read as [PAD]; None -> one [CLS] per row."""
    if prefix is None:
        return torch.full((B, 1), R.CLS, dtype=torch.int64)
    p = prefix.to(torch.int64).clone()
    return p.masked_fill(p == R.EOS, R.PAD)


class PrefixBeamState(BN.BlockedBeamState):
    """oracle/beam_ngram.py's ``BlockedBeamState`` for HF 4.16.2 ``beam_search`` with ``decoder_input_ids = prefix`` [B, P]
    (None = one [CLS] per row: exactly oracle/beam.py / oracle/beam_ngram.py).  All K beams of an image start from its prefix; a
    [SEP] inside it is read as [PAD], the in-place replacement ``decoder_forward`` applies before every forward
    (models/visual_dialog_decoder.py:53-57), and there is no decoder padding mask.  A hypothesis's length is its whole decoder
    input, P + t (HF's ``input_ids.shape[-1]``), in ``BeamHypotheses.add``, ``is_done`` and ``finalize``; the n-gram key of beam k is
    the last n-1 tokens of prefix_b + tokens[b, k, :t].  Every other piece of arithmetic is oracle/beam.py's.  The goldens pin only
    the [CLS] start: for longer prefixes this reading of the reference call site (models/visual_dialog_model.py:86-110, no decoder
    mask in decode mode) is the contract."""

    def __init__(self, B, K, V, max_new=18, prefix=None):
        super().__init__(B, K, V, max_new)
        self.prefix = decoder_input(prefix, B)
        self.P = self.prefix.shape[1]

    def banned(self, hist, n):
        return [R.ngram_banned_tokens(hist[b], self.prefix[b].tolist() + self.tokens[b, k, : self.t].tolist(), n) if n > 0 else []
                for b in range(self.B) for k in range(self.K)]

    def step(self, logits, ngram_blocking_size=0, hist=None):
        B, K, V = self.B, self.K, self.V
        cur_len = self.t + self.P
        sc = OB.candidate_scores(logits.float(), self.beam_scores)
        if ngram_blocking_size > 0:
            for row, toks in enumerate(self.banned(hist, ngram_blocking_size)):
                b, k = divmod(row, K)
                for w in toks:
                    sc[b, k * V + w] = -float("inf")
        val, idx = OB.top_candidates(sc, 2 * K)
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
                if tok == OB.EOS:
                    if rank >= K:
                        continue
                    self._add(b, self.tokens[b, beam, : self.t].tolist(), s.item(), cur_len)
                else:
                    nb_scores[b, n] = s; nb_tokens[b, n] = tok; nb_idx[b, n] = beam
                    n += 1
                if n == K:
                    break
            assert n == K
            if len(self.hyps[b]) >= K and self.worst[b] >= float(val[b].max().item()) / float(cur_len):
                self.done[b] = True
        new_tokens = self.tokens.gather(1, nb_idx[:, :, None].expand(-1, -1, self.T)).clone()
        new_tokens[:, :, self.t] = nb_tokens
        self.tokens, self.beam_scores = new_tokens, nb_scores
        self.last_beam_idx, self.last_tokens = nb_idx, nb_tokens
        self.t += 1
        return nb_idx, nb_tokens, nb_scores

    def finalize(self):
        B, T = self.B, self.T
        seq = torch.zeros(B, T, dtype=torch.int64)
        best_scores = torch.zeros(B, dtype=torch.float64)
        for b in range(B):
            if not self.done[b]:
                for k in range(self.K):
                    self._add(b, self.tokens[b, k, : self.t].tolist(), self.beam_scores[b, k].item(), self.t + self.P)
            score, toks = sorted(self.hyps[b], key=lambda x: x[0])[-1]
            seq[b, : len(toks)] = torch.tensor(toks, dtype=torch.int64)
            if len(toks) < T:
                seq[b, len(toks)] = OB.EOS
            best_scores[b] = score
        return seq, best_scores


def prefix_beam_search(sd, enc_cfg, dec_cfg, batch, num_beams=5, max_new=18, ngram_blocking_size=0, prefix=None):
    """oracle/beam_ngram.py:beam_search from the decoder prefix ``prefix`` (``PrefixBeamState``)."""
    ids, seg, att = batch["enc_input_ids"], batch["enc_segments"], batch["enc_att_mask"]
    B, K = ids.shape[0], num_beams
    seq_t, seq_v = R.encoder(sd, enc_cfg, ids, batch["enc_image_feat"], batch["enc_image_loc"], seg, att, batch["enc_image_mask"])
    enc_h, enc_m = R.vlfusion(sd, seq_t, seq_v, att, batch["enc_image_mask"])
    enc_h, enc_m = enc_h.repeat_interleave(K, 0), enc_m.repeat_interleave(K, 0)
    hist = BN.question_history(ids, seg)
    st = PrefixBeamState(B, K, dec_cfg.vocab_size, max_new, prefix)
    start = st.prefix.repeat_interleave(K, 0)
    for t in range(max_new):
        h = R.decoder_hidden(sd, dec_cfg, torch.cat((start, st.tokens.reshape(B * K, -1)[:, :t]), 1), None, enc_h, enc_m)
        st.step(R.lm_logits(sd, h[:, -1]), ngram_blocking_size, hist)
        if bool(st.done.all()):
            break
    return st.finalize()


def contains_banned_ngram(hist, seq, n, prefix):
    """True when prefix ([SEP] read as [PAD]) + seq holds an n-gram of ``hist`` that blocking would have banned."""
    toks = [R.PAD if int(x) == R.EOS else int(x) for x in prefix] + [int(x) for x in seq]
    bad = BN.banned_ngrams(hist, n)
    return any(tuple(toks[i:i + n]) in bad for i in range(len(toks) - n + 1))


# ---- CPU -----------------------------------------------------------------------------------------------------------
def test_beam_oracles_cls_prefix_equals_default(tiny_cfgs, tiny_sd):
    enc_cfg, dec_cfg = tiny_cfgs
    b = _with_question(history_batch(enc_cfg, 0, 2), A4["tiny"])
    sd = _with_bias(tiny_sd, {R.EOS: 2.5})
    cls = torch.full((2, 1), R.CLS, dtype=torch.int64)
    with torch.no_grad():
        for K in (3, 5):
            ref = OB.beam_search(sd, enc_cfg, dec_cfg, b, num_beams=K)
            for pre in (None, cls):
                got = prefix_beam_search(sd, enc_cfg, dec_cfg, b, num_beams=K, prefix=pre)
                assert torch.equal(ref[0], got[0]) and torch.equal(ref[1], got[1])
            for n in (0, 4):
                ref = BN.beam_search(sd, enc_cfg, dec_cfg, b, num_beams=K, ngram_blocking_size=n)
                for pre in (None, cls):
                    got = prefix_beam_search(sd, enc_cfg, dec_cfg, b, num_beams=K, ngram_blocking_size=n, prefix=pre)
                    assert torch.equal(ref[0], got[0]) and torch.equal(ref[1], got[1])
    # random logits: every step's (parent, token, score) and the finalised hypotheses
    g = torch.Generator().manual_seed(5)
    B, K, V, T = 3, 4, 160, 10
    logits = [torch.randn(B * K, V, generator=g) * 3 for _ in range(T)]
    for lg in logits[3:]:
        lg[:, OB.EOS] += 4.0
    st = OB.BeamState(B, K, V, T)
    ref = ([st.step(lg) for lg in logits], st.finalize())
    for pre in (None, torch.full((B, 1), R.CLS, dtype=torch.int64)):
        st = PrefixBeamState(B, K, V, T, prefix=pre)
        got = ([st.step(lg) for lg in logits], st.finalize())
        for a, c in zip(ref[0], got[0]):
            assert all(torch.equal(x, y) for x, y in zip(a, c))
        assert all(torch.equal(x, y) for x, y in zip(ref[1], got[1]))


@pytest.mark.parametrize("n", [3, 4])
def test_prefixed_blocked_oracle_never_selects_a_banned_token(n):
    g = torch.Generator().manual_seed(17 + n)
    B, K, V, T = 2, 3, 140, 8
    a, c = 120, 121
    hist = [[R.CLS, a, c, a, a, c, c, a, c, R.EOS, 0], [0, 130, a, a, a, c, a, 131, 0]]
    prefix = torch.tensor([[R.CLS, 9, a, c], [7, R.EOS, a, a]])          # keys of the first steps span the prefix
    logits = []
    for _ in range(T):
        lg = torch.randn(B * K, V, generator=g)
        lg[:, [a, c]] += 6.0
        lg[:, OB.EOS] -= 5.0
        logits.append(lg)
    st = PrefixBeamState(B, K, V, T, prefix=prefix)
    trace = [st.step(lg, n, hist) for lg in logits]
    seq, _ = st.finalize()
    free = PrefixBeamState(B, K, V, T, prefix=prefix)
    for lg in logits:
        free.step(lg)
    seq0, _ = free.finalize()
    tokens = torch.zeros(B, K, T, dtype=torch.int64)
    for t, (bi, bt, _) in enumerate(trace):
        for b in range(B):
            bad = BN.banned_ngrams(hist[b], n)
            for k in range(K):
                full = st.prefix[b].tolist() + tokens[b, bi[b, k], :t].tolist() + [int(bt[b, k])]
                assert tuple(full[-n:]) not in bad, (t, b, k, full)
        tokens = tokens.gather(1, bi[:, :, None].expand(-1, -1, T)).clone()
        tokens[:, :, t] = bt
    assert not any(contains_banned_ngram(hist[b], seq[b].tolist(), n, prefix[b]) for b in range(B))
    assert any(contains_banned_ngram(hist[b], seq0[b].tolist(), n, prefix[b]) for b in range(B)), "the unblocked run must copy a history n-gram"
    # the first step bans with keys that lie wholly inside the prefix ([SEP] read as [PAD] in row 1)
    assert st.prefix[1, 1] == R.PAD


def test_restatement_continues_its_own_greedy_output(tiny_cfgs, tiny_sd):
    enc_cfg, dec_cfg = tiny_cfgs
    b = history_batch(enc_cfg, 0, 3)
    g = _greedy_ref(tiny_sd, enc_cfg, dec_cfg, b, b["dec_input_ids"])
    for j in (1, 6):
        assert not (g[:, :j] == R.EOS).any()
        cont = _greedy_ref(tiny_sd, enc_cfg, dec_cfg, b, torch.cat((b["dec_input_ids"], g[:, :j]), 1), max_new=18 - j)
        assert torch.equal(cont, g[:, j:])


# ---- GPU: fp32 parity ----------------------------------------------------------------------------------------------
def _engine(enc_cfg, dec_cfg, sd, dtype, B, b, **kw):
    from gst_visdial_b200.engine import Engine
    e = Engine(enc_cfg, dec_cfg, dtype=dtype, max_batch=B, max_beams=5, **kw)
    e.load_state_dict(sd)
    o = e.encode(b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"], b["enc_image_mask"])
    e.prefill_cross(B, o["Le"])
    return e


def _hist(b):
    return dict(hist_ids=b["enc_input_ids"], hist_segments=b["enc_segments"])


@pytest.mark.gpu
@pytest.mark.parametrize("size", ["tiny", "full"])
def test_fp32_greedy_from_prefix_matches_restatement(size, tiny_cfgs, tiny_sd, full_cfgs, full_sd):
    enc_cfg, dec_cfg = tiny_cfgs if size == "tiny" else full_cfgs
    a, b4, c, d = A4[size]
    base = tiny_sd if size == "tiny" else full_sd
    B = 3 if size == "tiny" else 2
    b = _with_question(history_batch(enc_cfg, 0, B), A4[size])
    e = _engine(enc_cfg, dec_cfg, base, "fp32", B, b)
    try:
        for P in (2, 5, 15, 25):                                  # P = 25: 42 cached positions
            pre = _prefixes(B, P, enc_cfg.vocab_size)
            ref = _greedy_ref(base, enc_cfg, dec_cfg, b, pre)
            got = e.generate(B, num_beams=1, **_GREEDY, prefix=pre).cpu()
            assert torch.equal(got, ref), f"P={P}: {got.tolist()} vs {ref.tolist()}"
    finally:
        e.close()
    sd = _with_bias(base, {d: 30.0})
    e = _engine(enc_cfg, dec_cfg, sd, "fp32", B, b)
    try:
        # n = 4 with a prefix ending in the first three tokens of a history 4-gram: only a ban across the boundary stops the fourth
        pre = _prefixes(B, 8, enc_cfg.vocab_size)
        pre[:, -3:] = torch.tensor([a, b4, c])
        free = _greedy_ref(sd, enc_cfg, dec_cfg, b, pre, n=0)
        assert (free[:, 0] == d).all(), "precondition: without blocking the history 4-gram is completed"
        ref = _greedy_ref(sd, enc_cfg, dec_cfg, b, pre, n=4)
        assert (ref[:, 0] != d).all()
        for n, want in ((0, free), (4, ref)):
            got = e.generate(B, num_beams=1, **_GREEDY, ngram_blocking_size=n, prefix=pre, **_hist(b)).cpu()
            assert torch.equal(got, want), f"n={n}: {got.tolist()} vs {want.tolist()}"
    finally:
        e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["separate_calls", "whole_round", "no_cuda_graph"])
@pytest.mark.parametrize("n", [0, 4])
@pytest.mark.parametrize("K", [3, 5])
def test_tiny_fp32_prefixed_beams_match_oracle(tiny_cfgs, tiny_sd, K, n, path):
    from gst_visdial_b200 import _lib, weights as W
    from test_gpu_model import _build_model, _call
    enc_cfg, dec_cfg = tiny_cfgs
    a, b4, c, d = A4["tiny"]
    sd = _with_bias(tiny_sd, {R.EOS: 3.5, d: 3.0})             # hypotheses end early; the history 4-gram is attractive
    b = _with_question(history_batch(enc_cfg, 0, 3), A4["tiny"])
    pre = _prefixes(3, 6, enc_cfg.vocab_size)
    pre[0, -3:] = torch.tensor([a, b4, c])                        # the first step's key lies in the prefix
    pre[1, -2:] = torch.tensor([a, b4])                           # the second step's key spans the boundary
    with torch.no_grad():
        ref, ref_sc = prefix_beam_search(sd, enc_cfg, dec_cfg, b, num_beams=K, ngram_blocking_size=n, prefix=pre)
        if n == 0:
            assert (ref == R.EOS).any() and ref[0, 0] == d, "precondition: early hypotheses, and row 0 completes the 4-gram"
        else:
            assert ref[0, 0] != d
    kw = {"separate_calls": dict(engine_round_graph=False), "whole_round": {},
          "no_cuda_graph": dict(engine_flags=_lib.GSTVD_FLAG_NO_CUDA_GRAPH)}[path]
    model, _ = _build_model(W.TINY_ENC_CONFIG, W.TINY_DEC_CONFIG, sd, "fp32", **kw)
    seq, dec = _call(model, b, dec_ids=pre.clone(), ngram_blocking_size=n, num_beams=K, **_GREEDY)
    assert torch.equal(seq.cpu(), ref), f"{seq.cpu().tolist()} vs {ref.tolist()}"
    assert torch.equal(dec.cpu(), pre), "the caller's dec_input_ids must not be modified"
    eng = model.module._engine(torch.device("cuda:0"))
    seq2, sc2 = eng.generate(3, num_beams=K, ngram_blocking_size=n, prefix=pre, want_scores=True, **_hist(b))
    assert torch.equal(seq2.cpu(), ref)
    assert torch.allclose(sc2.cpu().double(), ref_sc, atol=1e-4), (sc2, ref_sc)


@pytest.mark.gpu
def test_tiny_fp32_single_non_cls_start_decodes(tiny_cfgs, tiny_sd):
    from gst_visdial_b200 import weights as W
    from test_gpu_model import _build_model, _call
    enc_cfg, dec_cfg = tiny_cfgs
    b = history_batch(enc_cfg, 0, 3)
    pre = torch.tensor([[7], [R.CLS], [R.EOS]])
    ref = _greedy_ref(tiny_sd, enc_cfg, dec_cfg, b, pre)
    for round_graph in (True, False):
        model, _ = _build_model(W.TINY_ENC_CONFIG, W.TINY_DEC_CONFIG, tiny_sd, "fp32", engine_round_graph=round_graph)
        seq, _ = _call(model, b, dec_ids=pre.clone(), ngram_blocking_size=0, **_GREEDY)
        assert torch.equal(seq.cpu(), ref)


# ---- GPU: bf16 product path ----------------------------------------------------------------------------------------
# Greedy from [CLS] + its own greedy output[:j] continues with output[j] on this share of the 64 rows or more.  bf16 rounding
# differs between the teacher-forced prefill and the decode steps, so a near-tie may flip; measured on an NVIDIA B200 (1000 W
# power limit): 0.984 (63 of 64 rows, j = 8).
CONTINUATION_MIN = 0.9


@pytest.mark.gpu
def test_full_bf16_prefix_paths_agree(full_cfgs, full_sd):
    from gst_visdial_b200 import _lib, weights as W
    from test_gpu_model import _build_model, _call
    enc_cfg, dec_cfg = full_cfgs
    B = 64
    b = history_batch(enc_cfg, 0, B)
    pre = _prefixes(B, 25, enc_cfg.vocab_size)                    # 42 cached positions
    modes = {"beam": dict(num_beams=5, **_GREEDY), "sample": dict(num_beams=1, temperature=0.7, top_k=7, top_p=0.0, seed=11)}
    outs = {}
    for name, kw in (("whole_round", {}), ("separate_calls", dict(engine_round_graph=False)),
                     ("no_cuda_graph", dict(engine_round_graph=False, engine_flags=_lib.GSTVD_FLAG_NO_CUDA_GRAPH))):
        model, _ = _build_model(W.DEFAULT_ENC_CONFIG, W.DEFAULT_DEC_CONFIG, full_sd, "bf16", engine_max_batch=B, **kw)
        for m, mk in modes.items():
            runs = [_call(model, b, dec_ids=pre.clone(), ngram_blocking_size=4, **mk)[0].cpu() for _ in range(2)]
            assert torch.equal(runs[0], runs[1]), f"{name} / {m}: repeated calls differ"
            outs[(name, m)] = runs[0]
        del model
        torch.cuda.empty_cache()
    for m in modes:
        assert torch.equal(outs[("separate_calls", m)], outs[("whole_round", m)]), f"{m}: whole-round graph differs from separate calls"
        assert torch.equal(outs[("no_cuda_graph", m)], outs[("whole_round", m)]), f"{m}: eager decode differs from the captured graph"

    e = _engine(enc_cfg, dec_cfg, full_sd, "bf16", B, b)
    try:
        cls = torch.full((B, 1), R.CLS, dtype=torch.int64)
        for mk in modes.values():
            kw = dict(mk, want_scores=True) if mk["num_beams"] > 1 else mk
            l0 = e.launch_count
            old = e.generate(B, **kw)
            l1 = e.launch_count
            new = e.generate(B, prefix=cls, **kw)
            l2 = e.launch_count
            old, new = (old, new) if isinstance(old, tuple) else ((old,), (new,))
            assert all(torch.equal(x, y) for x, y in zip(old, new)), "an explicit [CLS] prefix differs from the implicit [CLS] start"
            assert l1 - l0 == l2 - l1
        g = e.generate(B, num_beams=1, **_GREEDY).cpu()
        j = 8
        first = e.generate(B, num_beams=1, **_GREEDY, prefix=torch.cat((cls, g[:, :j]), 1)).cpu()[:, 0]
        live = ~(g[:, :j] == R.EOS).any(1)
        agree = (first[live] == g[live, j]).float().mean().item()
        print(f"greedy continuation agreement at the first generated position: {agree:.3f} over {int(live.sum())} rows")
        assert agree >= CONTINUATION_MIN, agree
    finally:
        e.close()


# ---- GPU: argument checks ------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_prefix_rejections(tiny_cfgs, tiny_sd):
    from gst_visdial_b200 import _lib, weights as W
    from gst_visdial_b200._lib import GstvdError
    enc_cfg, dec_cfg = tiny_cfgs
    B = 2
    b = history_batch(enc_cfg, 0, B)
    e = _engine(enc_cfg, dec_cfg, tiny_sd, "fp32", B, b, max_dec_len=60)
    try:
        with pytest.raises(GstvdError):
            e.generate(B, prefix=torch.zeros(B, 0, dtype=torch.int64))              # P < 1
        with pytest.raises(GstvdError):
            e.generate(B, prefix=torch.full((B, 61), R.CLS))                          # P > max_dec_len
        with pytest.raises(GstvdError):
            e.generate(B, prefix=torch.full((B, 48), R.CLS))                          # 47 + 18 > 64 cached positions
        e.generate(B, prefix=torch.full((B, 47), R.CLS))                              # 64: accepted
        gp = _lib.GstvdGenParams()
        gp.mode, gp.num_beams, gp.max_new_tokens, gp.top_k, gp.temperature = _lib.GSTVD_SELECT_SAMPLE, 1, 18, 1, 1.0
        gp.num_return_sequences = gp.num_beam_groups = 1
        out = torch.empty(B, 18, dtype=torch.int64, device="cuda:0")
        rc = e.lib.gstvd_generate(e.ctx, B, ctypes.byref(gp), None, 3, None, None, 0, ctypes.c_void_p(out.data_ptr()), None, e._stream())
        with pytest.raises(GstvdError):
            _lib.check(e.ctx, rc)                                                     # NULL prefix with P > 1
        with pytest.raises(GstvdError):
            e.round(b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"], b["enc_image_mask"],
                    prefix=torch.full((B, 61), R.CLS))
    finally:
        e.close()
    # P - 1 + max_new_tokens above max_position_embeddings
    enc32, dec32 = copy.deepcopy(enc_cfg), copy.deepcopy(dec_cfg)
    enc32.max_position_embeddings = dec32.max_position_embeddings = 32
    sd32 = W.synthetic_state_dict(enc32, dec32, seed=0)
    from gst_visdial_b200.engine import Engine
    e = Engine(enc32, dec32, dtype="fp32", max_batch=B, max_beams=5, max_text_len=16)
    try:
        e.load_state_dict(sd32)
        e.prefill_cross(B, 8, torch.randn(B, 8, enc32.hidden_size))

        e.generate(B, prefix=torch.full((B, 15), R.CLS))                              # 14 + 18 = 32: accepted
        with pytest.raises(GstvdError):
            e.generate(B, prefix=torch.full((B, 16), R.CLS))
    finally:
        e.close()
