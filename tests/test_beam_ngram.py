"""Beam search with question-history n-gram blocking (the questioner's decoding, generate.py:124, with beams).

CPU: the blocked beam oracle (oracle/beam_ngram.py) reduces to oracle/beam.py at n = 0 and never selects a banned (beam, token);
the -q_num_beams flag.  GPU: the engine's ids are identical to the oracle in fp32 on every call path, and the bf16 product path
returns no banned n-gram, agrees across call paths and is deterministic.

Random weights rarely repeat a history n-gram, so the GPU cases raise the LM-head bias of two tokens and put a de Bruijn sequence
of them (every n-gram over the two, n <= 4) into a question segment of the history: unblocked beams then copy history n-grams,
which the tests assert first so that they cannot pass without a ban taking effect.
"""
import os

import pytest
import torch

from helpers import R, history_batch
from oracle import beam as OB
from oracle import beam_ngram as BN

# de Bruijn sequence B(2, 4) over {a, b}, linearised: holds every 4-gram (hence every 2- and 3-gram) over the two tokens
_DE_BRUIJN = (0, 0, 0, 0, 1, 0, 0, 1, 1, 0, 1, 0, 1, 1, 1, 1, 0, 0, 0)


def _boosted(sd, toks, add=5.0):
    sd = dict(sd)
    bias = sd["decoder.decoder.lm_head.bias"].clone()
    bias[list(toks)] += add
    sd["decoder.decoder.lm_head.bias"] = bias
    sd["decoder.decoder.lm_head.decoder.bias"] = bias
    return sd


def _with_question(b, toks):
    """Splices the de Bruijn sequence over ``toks`` (+ [SEP]) into every row's history as a question (segment 0)."""
    ids, seg = b["enc_input_ids"], b["enc_segments"]
    utt = torch.tensor([toks[i] for i in _DE_BRUIJN] + [R.EOS]).repeat(ids.shape[0], 1)
    R.splice(ids, seg, (ids != 0).sum(-1), utt, None, set())
    b["enc_att_mask"] = (ids != 0).float()
    return b


def _hits(b, seq, n):
    hist = BN.question_history(b["enc_input_ids"], b["enc_segments"])
    return [BN.contains_banned_ngram(hist[i], seq[i].tolist(), n) for i in range(seq.shape[0])]


# ---- CPU: oracle ---------------------------------------------------------------------------------------------------
def _random_run(state_cls, logits_seq, B, K, V, **step_kw):
    st = state_cls(B, K, V, len(logits_seq))
    trace = [st.step(lg, **step_kw) for lg in logits_seq]
    seq, sc = st.finalize()
    return st, trace, seq, sc


def test_blocked_oracle_without_blocking_equals_beam_oracle(tiny_cfgs, tiny_sd):
    g = torch.Generator().manual_seed(3)
    B, K, V, T = 3, 4, 160, 12
    logits = [torch.randn(B * K, V, generator=g) * 3 for _ in range(T)]
    for lg in logits[4:]:
        lg[:, OB.EOS] += 4.0                                   # hypotheses, early finish and padded images
    _, tr0, s0, c0 = _random_run(OB.BeamState, logits, B, K, V)
    _, tr1, s1, c1 = _random_run(BN.BlockedBeamState, logits, B, K, V, ngram_blocking_size=0)
    for a, b in zip(tr0, tr1):
        assert all(torch.equal(x, y) for x, y in zip(a, b))
    assert torch.equal(s0, s1) and torch.equal(c0, c1)
    enc_cfg, dec_cfg = tiny_cfgs
    b = history_batch(enc_cfg, 0, 2)
    with torch.no_grad():
        ref, ref_sc = OB.beam_search(tiny_sd, enc_cfg, dec_cfg, b, num_beams=5)
        got, got_sc = BN.beam_search(tiny_sd, enc_cfg, dec_cfg, b, num_beams=5, ngram_blocking_size=0)
    assert torch.equal(ref, got) and torch.equal(ref_sc, got_sc)


@pytest.mark.parametrize("n", [2, 3])
def test_blocked_oracle_never_selects_a_banned_token(n):
    g = torch.Generator().manual_seed(11 + n)
    B, K, V, T = 2, 3, 140, 10
    a, c = 120, 121
    hist = [[R.CLS] + [[a, c][i] for i in _DE_BRUIJN] + [R.EOS] + [0] * 5, [0, 130, 131, 132, 133, a, c, a, a, c, c, 0]]
    logits = []
    for _ in range(T):
        lg = torch.randn(B * K, V, generator=g)
        lg[:, [a, c]] += 6.0
        lg[:, OB.EOS] -= 5.0
        logits.append(lg)
    st, trace, seq, _ = _random_run(BN.BlockedBeamState, logits, B, K, V, ngram_blocking_size=n, hist=hist)
    _, _, seq0, _ = _random_run(OB.BeamState, logits, B, K, V)
    # replay the selections: every (parent beam, token) pair must not complete a history n-gram of the parent's prefix
    tokens = torch.zeros(B, K, T, dtype=torch.int64)
    for t, (bi, bt, _) in enumerate(trace):
        for b in range(B):
            bad = BN.banned_ngrams(hist[b], n)
            for k in range(K):
                prefix = [R.CLS] + tokens[b, bi[b, k], :t].tolist() + [int(bt[b, k])]
                assert tuple(prefix[-n:]) not in bad, (t, b, k, prefix)
        tokens = tokens.gather(1, trace[t][0][:, :, None].expand(-1, -1, T)).clone()
        tokens[:, :, t] = trace[t][1]
    assert torch.equal(tokens, st.tokens)
    assert not any(BN.contains_banned_ngram(hist[b], seq[b].tolist(), n) for b in range(B))
    assert any(BN.contains_banned_ngram(hist[b], seq0[b].tolist(), n) for b in range(B)), "the unblocked run must copy a history n-gram"
    assert not torch.equal(seq, seq0)


def test_q_num_beams_option(tmp_path):
    from gst_visdial_b200 import options
    base = ["-save_path", str(tmp_path)]
    p = options.read_command_line(base)
    assert p["q_num_beams"] == 1 and p["engine_max_beams"] == 1
    p = options.read_command_line(base + ["-q_num_beams", "5"])
    assert p["q_num_beams"] == 5 and p["num_beams"] == 1 and p["engine_max_beams"] == 5
    p = options.read_command_line(base + ["-num_beams", "3", "-q_num_beams", "2"])
    assert p["engine_max_beams"] == 3


# ---- GPU -----------------------------------------------------------------------------------------------------------
TINY_TOKS = (500, 501)
FULL_TOKS = (2000, 2001)
_Q = dict(temperature=1.0, top_k=1, top_p=0.0)


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["separate_calls", "whole_round", "no_cuda_graph"])
@pytest.mark.parametrize("n", [2, 4])
def test_tiny_fp32_blocked_beams_match_oracle(tiny_cfgs, tiny_sd, n, path):
    from gst_visdial_b200 import _lib, weights as W
    from test_gpu_model import _build_model, _call
    enc_cfg, dec_cfg = tiny_cfgs
    sd = _boosted(tiny_sd, TINY_TOKS)
    b = _with_question(history_batch(enc_cfg, 0, 3), TINY_TOKS)
    with torch.no_grad():
        ref0, _ = OB.beam_search(sd, enc_cfg, dec_cfg, b, num_beams=5)
        ref, _ = BN.beam_search(sd, enc_cfg, dec_cfg, b, num_beams=5, ngram_blocking_size=n)
    assert all(_hits(b, ref0, n)), "precondition: the unblocked beams must copy a history n-gram"
    assert not any(_hits(b, ref, n))
    kw = {"separate_calls": dict(engine_round_graph=False), "whole_round": {},
          "no_cuda_graph": dict(engine_flags=_lib.GSTVD_FLAG_NO_CUDA_GRAPH)}[path]
    model, _ = _build_model(W.TINY_ENC_CONFIG, W.TINY_DEC_CONFIG, sd, "fp32", **kw)
    seq, _ = _call(model, b, ngram_blocking_size=n, num_beams=5, **_Q)
    assert torch.equal(seq.cpu(), ref), f"{seq.cpu().tolist()} vs {ref.tolist()}"
    seq0, _ = _call(model, b, ngram_blocking_size=0, num_beams=5, **_Q)      # same context, blocking off again
    assert torch.equal(seq0.cpu(), ref0)


@pytest.fixture(scope="module")
def full_boosted(full_sd):
    return _boosted(full_sd, FULL_TOKS)


@pytest.mark.gpu
def test_full_fp32_blocked_beams_match_oracle(full_cfgs, full_boosted):
    from gst_visdial_b200.engine import Engine
    enc_cfg, dec_cfg = full_cfgs
    b = _with_question(history_batch(enc_cfg, 0, 2), FULL_TOKS)
    with torch.no_grad():
        seq_t, seq_v = R.encoder(full_boosted, enc_cfg, b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"],
                                 b["enc_att_mask"], b["enc_image_mask"])
        ref, ref_sc = BN.beam_search(full_boosted, enc_cfg, dec_cfg, b, num_beams=5, ngram_blocking_size=4, precomputed_encoder=(seq_t, seq_v))
    e = Engine(enc_cfg, dec_cfg, dtype="fp32", max_batch=2, max_beams=5)
    try:
        e.load_state_dict(full_boosted)
        o = e.encode(b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"], b["enc_image_mask"])
        e.prefill_cross(2, o["Le"])
        seq, sc = e.generate(2, num_beams=5, ngram_blocking_size=4, hist_ids=b["enc_input_ids"], hist_segments=b["enc_segments"],
                             want_scores=True)
        assert torch.equal(seq.cpu(), ref), f"{seq.cpu().tolist()} vs {ref.tolist()}"
        assert torch.allclose(sc.cpu().double(), ref_sc, atol=1e-3)
    finally:
        e.close()


@pytest.mark.gpu
def test_full_bf16_blocked_beams_paths_agree(full_cfgs, full_boosted):
    from gst_visdial_b200 import _lib, weights as W
    from test_gpu_model import _build_model, _call
    enc_cfg, _ = full_cfgs
    b = _with_question(history_batch(enc_cfg, 0, 8), FULL_TOKS)
    outs = {}
    for name, kw in (("whole_round", {}), ("separate_calls", dict(engine_round_graph=False)),
                     ("no_cuda_graph", dict(engine_round_graph=False, engine_flags=_lib.GSTVD_FLAG_NO_CUDA_GRAPH))):
        model, _ = _build_model(W.DEFAULT_ENC_CONFIG, W.DEFAULT_DEC_CONFIG, full_boosted, "bf16", **kw)
        if name == "whole_round":
            seq0 = _call(model, b, ngram_blocking_size=0, num_beams=5, **_Q)[0].cpu()
            assert any(_hits(b, seq0, 4)), "precondition: the unblocked beams must copy a history n-gram"
        runs = [_call(model, b, ngram_blocking_size=4, num_beams=5, **_Q)[0].cpu() for _ in range(2)]
        assert torch.equal(runs[0], runs[1]), f"{name}: repeated calls differ"
        outs[name] = runs[0]
        del model
        torch.cuda.empty_cache()
    seq = outs["whole_round"]
    assert not any(_hits(b, seq, 4)), seq.tolist()
    assert not torch.equal(seq, seq0)
    assert torch.equal(outs["separate_calls"], seq), "whole-round graph differs from separate calls"
    assert torch.equal(outs["no_cuda_graph"], seq), "eager decode differs from the captured graph"


@pytest.mark.gpu
def test_full_bf16_dialog_loop_blocked_question_beams(full_cfgs, full_sd, full_boosted):
    from gst_visdial_b200 import weights as W
    from gst_visdial_b200.dialog import generate_dialogs
    from test_gpu_model import _build_model
    enc_cfg, _ = full_cfgs
    B, rounds = 4, 2
    b = _with_question(history_batch(enc_cfg, 0, B, rounds=1), FULL_TOKS)
    q_model, _ = _build_model(W.DEFAULT_ENC_CONFIG, W.DEFAULT_DEC_CONFIG, full_boosted, "bf16", model="enc_dec_q")
    a_model, _ = _build_model(W.DEFAULT_ENC_CONFIG, W.DEFAULT_DEC_CONFIG, full_sd, "bf16", model="enc_dec_a")
    q_kwargs = dict(num_beams=5, ngram_blocking_size=4, temperature=0.7, top_k=7, top_p=0.0)
    res = generate_dialogs(a_model, b, q_model=q_model, num_rounds=rounds, q_kwargs=q_kwargs, with_ppl=True, device="cuda:0")
    free = generate_dialogs(a_model, b, q_model=q_model, num_rounds=1, q_kwargs=dict(q_kwargs, ngram_blocking_size=0), with_ppl=False,
                            device="cuda:0")
    assert any(_hits(b, free.questions[:, 0].cpu(), 4)), "precondition: unblocked question beams must copy a history n-gram"
    # replay the splices on the host: each question is checked against the history as it stood before it was spliced in
    ids, seg = b["enc_input_ids"].clone(), b["enc_segments"].clone()
    enc_len = (ids != 0).sum(-1)
    for r in range(rounds):
        q, a = res.questions[:, r].cpu(), res.answers[:, r].cpu()
        assert not any(_hits(dict(enc_input_ids=ids, enc_segments=seg), q, 4)), f"round {r}: {q.tolist()}"
        enc_len = enc_len + R.splice(ids, seg, enc_len, q, None, set())
        enc_len = enc_len + R.splice(ids, seg, enc_len, a.masked_fill(a == R.EOS, 0), 1, set())
    assert torch.equal(ids, res.enc_input_ids.cpu())


@pytest.mark.gpu
def test_generate_cli_question_beams(tmp_path):
    import json
    import subprocess
    import sys
    from helpers import ROOT
    cmd = [sys.executable, os.path.join(ROOT, "generate.py"), "-synthetic", "8", "-batch_size", "8", "-num_beams", "5", "-q_num_beams", "5",
           "-num_rounds", "2", "-save_path", str(tmp_path), "-save_name", "o.json"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout + r.stderr
    out = json.load(open(tmp_path / "o.json"))
    assert len(out) == 8 and all(len(d["dialog"]) == 2 for d in out)
