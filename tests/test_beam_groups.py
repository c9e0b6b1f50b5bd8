"""Diverse beam search: beam groups with a Hamming diversity penalty (include/gstvd.h gstvd_generate, params.num_beam_groups /
params.diversity_penalty; contract in oracle/beam_groups.py).

CPU: the group oracle with one group is the plain / blocked / prefixed beam oracle for any penalty; with G = K and no penalty every
group is greedy; with a large penalty and groups of one beam the groups take pairwise distinct tokens; an image that group 0 finishes
mid-step adds nothing from the later groups; the four CLI flags.
GPU: ids identical to the oracle (scores within 1e-4) in fp32 on every call path, with and without blocking and a decoder prefix, at
tiny and full size; G = K without penalty returns K copies of the greedy sample; the bf16 product path agrees across call paths, G = 1
gives the same ids, scores and launch count with and without a penalty, and the penalty separates the beams of every image; the
dialog loop and generate.py run with groups; every rejected argument raises.
"""
import copy
import os

import pytest
import torch

from helpers import R, history_batch
from oracle import beam as OB
from oracle import beam_ngram as BN
from oracle.beam_groups import GroupBeamState, group_beam_state
from oracle.beam_nbest import finalize_nbest
from test_beam_ngram import FULL_TOKS, TINY_TOKS, _boosted, _hits
from test_beam_ngram import _with_question as _with_de_bruijn
from test_decoder_prefix import PrefixBeamState, _prefixes

_GREEDY = dict(temperature=1.0, top_k=1, top_p=0.0)


def _random_logits(B, K, V, T, seed, eos_from=3):
    g = torch.Generator().manual_seed(seed)
    logits = [torch.randn(B * K, V, generator=g) * 3 for _ in range(T)]
    for lg in logits[eos_from:]:
        lg[:, OB.EOS] += 4.0
    return logits


def _same_steps(a, b):
    return all(torch.equal(x, y) for s, t in zip(a, b) for x, y in zip(s, t)) and len(a) == len(b)


# ---- CPU: oracle ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("lam", [0.0, 0.5, 3.0])
def test_group_oracle_one_group_is_beam_search(lam):
    B, K, V, T = 3, 4, 160, 10
    a, c = 120, 121
    hist = [[R.CLS, a, c, a, a, c, c, a, c, R.EOS], [0, 130, a, a, c, a, 131, 0], [a, c, a, c, c]]
    prefix = torch.tensor([[R.CLS, 9, a, c, 11], [7, R.EOS, a, a, 12], [R.CLS, R.CLS, R.CLS, c, a]])
    logits = _random_logits(B, K, V, T, seed=7)
    for lg in logits:
        lg[:, [a, c]] += 3.0
    cases = [(lambda: OB.BeamState(B, K, V, T), None, 0), (lambda: BN.BlockedBeamState(B, K, V, T), None, 4),
             (lambda: PrefixBeamState(B, K, V, T, prefix=prefix), prefix, 0), (lambda: PrefixBeamState(B, K, V, T, prefix=prefix), prefix, 4)]
    for make, pre, n in cases:
        kw = dict(ngram_blocking_size=n, hist=hist) if n else {}
        ref, got = make(), GroupBeamState(B, K, V, T, num_beam_groups=1, diversity_penalty=lam, prefix=pre)
        ref_steps = [ref.step(lg, **kw) for lg in logits]
        got_steps = [got.step(lg, **kw) for lg in logits]
        assert _same_steps(ref_steps, got_steps), (pre is not None, n)
        assert ref.hyps == got.hyps and torch.equal(ref.done, got.done)
        for N in (1, 2, K):
            r, g = finalize_nbest(copy.deepcopy(ref), N), finalize_nbest(copy.deepcopy(got), N)
            assert torch.equal(r[0], g[0]) and torch.equal(r[1], g[1]), N
        r, g = ref.finalize(), got.finalize()
        assert torch.equal(r[0], g[0]) and torch.equal(r[1], g[1])


def test_group_oracle_without_penalty_every_group_is_greedy():
    B, K, V, T = 2, 4, 150, 8
    g = torch.Generator().manual_seed(3)
    rows = [torch.randn(B, V, generator=g) * 3 for _ in range(T)]
    for t in range(T):
        rows[t][:, OB.EOS] = -50.0
    rows[5][0, OB.EOS] = 50.0                                       # image 0 ends after 5 tokens, image 1 runs to the end
    st = GroupBeamState(B, K, V, T, num_beam_groups=K, diversity_penalty=0.0)
    for t in range(T):
        if bool(st.done.all()):
            break
        st.step(rows[t].repeat_interleave(K, 0))                    # every beam of an image sees the image's row
    seq, _ = finalize_nbest(st, K)
    for b in range(B):
        greedy = []
        for t in range(T):
            w = int(rows[t][b].argmax())
            if w == OB.EOS:
                break
            greedy.append(w)
        want = torch.zeros(T, dtype=torch.int64)
        want[:len(greedy)] = torch.tensor(greedy)
        if len(greedy) < T:
            want[len(greedy)] = OB.EOS
        assert len(greedy) == (5 if b == 0 else T)
        assert all(torch.equal(seq[b * K + k], want) for k in range(K)), (b, seq[b * K: (b + 1) * K].tolist(), want.tolist())


def test_group_oracle_large_penalty_separates_the_groups():
    B, K, V, T = 3, 4, 150, 10
    g = torch.Generator().manual_seed(9)
    logits = [torch.randn(B, V, generator=g).repeat_interleave(K, 0) * 3 for _ in range(T)]   # the beams of an image agree
    for lg in logits:
        lg[:, OB.EOS] = -50.0
    st = GroupBeamState(B, K, V, T, num_beam_groups=K, diversity_penalty=1e4)
    checked = 0
    for lg in logits:
        _, tok, _ = st.step(lg)
        for b in range(B):
            if not st.done[b]:
                assert len(set(tok[b].tolist())) == K, (st.t, b, tok[b].tolist())
                checked += 1
    assert checked == B * T
    free = GroupBeamState(B, K, V, T, num_beam_groups=K, diversity_penalty=0.0)
    toks = [free.step(lg)[1] for lg in logits]
    assert all(len(set(tok[b].tolist())) == 1 for tok in toks for b in range(B)), "without the penalty every group takes the argmax"


def test_group_oracle_image_done_mid_step():
    """K = 2 beams in G = 2 groups.  Step 1: group 0 closes its second hypothesis; the heap (capacity K = 2) is full and no candidate
    of the group can improve it, so the image is done.  Group 1's best candidate at that step is an [SEP] whose hypothesis would
    displace the worst one, but HF tests ``done`` before every group's process: it must not be added, and group 1 is padded."""
    B, K, V, T = 1, 2, 200, 4

    def row(best, second, gap):
        r = torch.full((V,), -20.0)
        r[best], r[second] = 0.0, -gap
        return r
    steps = [torch.stack([row(OB.EOS, 5, 1.5), row(6, 7, 1.0)]),   # group 0: [SEP] first (hypothesis []), beam 5; group 1: beam 6
             torch.stack([row(OB.EOS, 8, 3.0), row(OB.EOS, 9, 3.0)])]
    st = GroupBeamState(B, K, V, T, num_beam_groups=2, diversity_penalty=0.5)
    st.step(steps[0])
    assert not st.done[0] and [h[1] for h in st.hyps[0]] == [[]]
    idx, tok, sc = st.step(steps[1])
    assert bool(st.done[0])
    assert [h[1] for h in st.hyps[0]] == [[], [5]], st.hyps[0]
    group1_sep = float(torch.log_softmax(steps[1][1], -1)[OB.EOS]) + float(torch.log_softmax(steps[0][1], -1)[6])
    assert group1_sep / 2 > st.worst[0], "precondition: group 1's [SEP] would enter the heap if it were processed"
    assert tok[0, 1] == R.PAD and sc[0, 1] == 0.0 and idx[0, 1] == 1
    seq, _ = finalize_nbest(st, K)
    assert seq[:, :2].tolist() == [[OB.EOS, 0], [5, OB.EOS]]


def test_group_oracle_rejects_bad_groups():
    for G, lam in ((0, 0.0), (3, 0.0), (2, -1.0), (2, float("nan")), (2, float("inf"))):
        with pytest.raises(ValueError):
            GroupBeamState(1, 4, 100, 5, num_beam_groups=G, diversity_penalty=lam)


def test_beam_group_options(tmp_path):
    from gst_visdial_b200 import options
    base = ["-save_path", str(tmp_path)]
    p = options.read_command_line(base)
    assert (p["num_beam_groups"], p["diversity_penalty"], p["q_num_beam_groups"], p["q_diversity_penalty"]) == (1, 0.0, 1, 0.0)
    p = options.read_command_line(base + ["-num_beams", "6", "-num_beam_groups", "3", "-diversity_penalty", "0.5",
                                          "-q_num_beams", "4", "-q_num_beam_groups", "4", "-q_diversity_penalty", "1.5"])
    assert (p["num_beam_groups"], p["diversity_penalty"], p["q_num_beam_groups"], p["q_diversity_penalty"]) == (3, 0.5, 4, 1.5)
    assert p["engine_max_beams"] == 6
    for bad in (["-num_beams", "6", "-num_beam_groups", "4"], ["-num_beam_groups", "2"], ["-q_num_beams", "5", "-q_num_beam_groups", "2"],
                ["-q_num_beam_groups", "3"], ["-num_beams", "4", "-num_beam_groups", "0"], ["-num_beams", "4", "-diversity_penalty", "-1"],
                ["-q_num_beams", "4", "-q_diversity_penalty", "inf"]):
        with pytest.raises(SystemExit):
            options.read_command_line(base + bad)


# ---- GPU: fp32 against the oracle ----------------------------------------------------------------------------------
_ORACLE = {}


def _oracle(sd, enc_cfg, dec_cfg, b, K, G, lam, n, prefix=None, Ns=(1,), tag=""):
    key = (tag, K, G, lam, n, prefix is not None)
    if key not in _ORACLE:
        with torch.no_grad():
            st = group_beam_state(sd, enc_cfg, dec_cfg, b, K, G, lam, ngram_blocking_size=n, prefix=prefix)
        _ORACLE[key] = {N: finalize_nbest(copy.deepcopy(st), N) for N in range(1, K + 1)}
    return {N: _ORACLE[key][N] for N in Ns}


def _hist(b):
    return dict(hist_ids=b["enc_input_ids"], hist_segments=b["enc_segments"])


def _path_kw(path):
    from gst_visdial_b200 import _lib
    return {"separate_calls": dict(engine_round_graph=False), "whole_round": {},
            "no_cuda_graph": dict(engine_flags=_lib.GSTVD_FLAG_NO_CUDA_GRAPH)}[path]


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["separate_calls", "whole_round", "no_cuda_graph"])
@pytest.mark.parametrize("n", [0, 4])
@pytest.mark.parametrize("lam", [0.0, 0.5])
@pytest.mark.parametrize("K,G", [(4, 2), (6, 3), (6, 6)])
def test_tiny_fp32_group_beams_match_oracle(tiny_cfgs, tiny_sd, K, G, lam, n, path):
    from gst_visdial_b200 import weights as W
    from test_gpu_model import _build_model, _call
    enc_cfg, dec_cfg = tiny_cfgs
    sd = _boosted(tiny_sd, TINY_TOKS)
    sd["decoder.decoder.lm_head.bias"][R.EOS] += 5.0             # hypotheses end early and compete for the shared heap
    b = _with_de_bruijn(history_batch(enc_cfg, 0, 3), TINY_TOKS)
    refs = _oracle(sd, enc_cfg, dec_cfg, b, K, G, lam, n, Ns=(1, K), tag="tiny")
    free = _oracle(sd, enc_cfg, dec_cfg, b, K, G, lam, 0, Ns=(1,), tag="tiny")[1][0]
    assert any(_hits(b, free, 4)), "precondition: the unblocked beams copy a history 4-gram"
    if n:
        assert not any(_hits(b, refs[1][0], 4))
    assert (refs[K][0] == R.EOS).any(), "precondition: some hypotheses end before the last step"
    model, _ = _build_model(W.TINY_ENC_CONFIG, W.TINY_DEC_CONFIG, sd, "fp32", engine_max_beams=6, **_path_kw(path))
    eng = model.module._engine(torch.device("cuda:0"))
    gk = dict(num_beams=K, num_beam_groups=G, diversity_penalty=lam, ngram_blocking_size=n)
    for N, (ref, ref_sc) in refs.items():
        seq, _ = _call(model, b, num_return_sequences=N, **gk, **_GREEDY)
        assert torch.equal(seq.cpu(), ref), f"N={N}: {seq.cpu().tolist()} vs {ref.tolist()}"
        seq2, sc2 = eng.generate(3, want_scores=True, num_return_sequences=N, **gk, **_hist(b))
        assert torch.equal(seq2.cpu(), ref)
        assert torch.allclose(sc2.cpu().double(), ref_sc, atol=1e-4), (sc2, ref_sc)


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["separate_calls", "whole_round", "no_cuda_graph"])
def test_tiny_fp32_group_beams_from_prefix_match_oracle(tiny_cfgs, tiny_sd, path):
    from gst_visdial_b200 import weights as W
    from test_gpu_model import _build_model, _call
    enc_cfg, dec_cfg = tiny_cfgs
    K, G, lam, n = 6, 3, 0.5, 4
    sd = _boosted(tiny_sd, TINY_TOKS)
    b = _with_de_bruijn(history_batch(enc_cfg, 0, 3), TINY_TOKS)
    pre = _prefixes(3, 5, enc_cfg.vocab_size)
    pre[0, -3:] = torch.tensor([TINY_TOKS[0]] * 3)                 # the first step's key lies in the prefix
    refs = _oracle(sd, enc_cfg, dec_cfg, b, K, G, lam, n, prefix=pre, Ns=(1, K), tag="tiny")
    model, _ = _build_model(W.TINY_ENC_CONFIG, W.TINY_DEC_CONFIG, sd, "fp32", engine_max_beams=6, **_path_kw(path))
    eng = model.module._engine(torch.device("cuda:0"))
    gk = dict(num_beams=K, num_beam_groups=G, diversity_penalty=lam, ngram_blocking_size=n)
    for N, (ref, ref_sc) in refs.items():
        seq, dec = _call(model, b, dec_ids=pre.clone(), num_return_sequences=N, **gk, **_GREEDY)
        assert torch.equal(seq.cpu(), ref), f"N={N}: {seq.cpu().tolist()} vs {ref.tolist()}"
        assert torch.equal(dec.cpu(), pre)
        seq2, sc2 = eng.generate(3, want_scores=True, num_return_sequences=N, prefix=pre, **gk, **_hist(b))
        assert torch.equal(seq2.cpu(), ref)
        assert torch.allclose(sc2.cpu().double(), ref_sc, atol=1e-4), (sc2, ref_sc)


def _engine(enc_cfg, dec_cfg, sd, dtype, b, **kw):
    from gst_visdial_b200.engine import Engine
    B = b["enc_input_ids"].shape[0]
    kw.setdefault("max_beams", 6)
    e = Engine(enc_cfg, dec_cfg, dtype=dtype, max_batch=B, **kw)
    e.load_state_dict(sd)
    o = e.encode(b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"], b["enc_image_mask"])
    e.prefill_cross(B, o["Le"])
    return e


@pytest.mark.gpu
def test_full_fp32_group_beams_match_oracle(full_cfgs, full_sd):
    enc_cfg, dec_cfg = full_cfgs
    K, G, lam, n = 6, 3, 0.5, 4
    sd = _boosted(full_sd, FULL_TOKS)
    b = _with_de_bruijn(history_batch(enc_cfg, 0, 2), FULL_TOKS)
    refs = _oracle(sd, enc_cfg, dec_cfg, b, K, G, lam, n, Ns=(1, K), tag="full")
    e = _engine(enc_cfg, dec_cfg, sd, "fp32", b)
    try:
        for N, (ref, ref_sc) in refs.items():
            seq, sc = e.generate(2, num_beams=K, num_beam_groups=G, diversity_penalty=lam, ngram_blocking_size=n, want_scores=True,
                                 num_return_sequences=N, **_hist(b))
            assert torch.equal(seq.cpu(), ref), f"N={N}: {seq.cpu().tolist()} vs {ref.tolist()}"
            assert torch.allclose(sc.cpu().double(), ref_sc, atol=1e-4)
    finally:
        e.close()


@pytest.mark.gpu
def test_fp32_groups_without_penalty_are_greedy(tiny_cfgs, tiny_sd):
    enc_cfg, dec_cfg = tiny_cfgs
    B, K = 3, 6
    b = history_batch(enc_cfg, 0, B)
    e = _engine(enc_cfg, dec_cfg, tiny_sd, "fp32", b)
    try:
        greedy = e.generate(B, num_beams=1, **_GREEDY).cpu()
        seq = e.generate(B, num_beams=K, num_beam_groups=K, diversity_penalty=0.0, num_return_sequences=K).cpu()
        assert torch.equal(seq, greedy.repeat_interleave(K, 0)), f"{seq.tolist()} vs {greedy.tolist()}"
    finally:
        e.close()


# ---- GPU: bf16 product path ----------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_full_bf16_group_beams(full_cfgs, full_sd):
    from gst_visdial_b200 import _lib, weights as W
    from test_gpu_model import _build_model, _call
    enc_cfg, dec_cfg = full_cfgs
    B, K = 64, 6
    b = history_batch(enc_cfg, 0, B)
    gk = dict(num_beams=K, num_beam_groups=3, diversity_penalty=0.5, ngram_blocking_size=4, num_return_sequences=K, **_GREEDY)
    outs = {}
    for name, kw in (("whole_round", {}), ("separate_calls", dict(engine_round_graph=False)),
                     ("no_cuda_graph", dict(engine_round_graph=False, engine_flags=_lib.GSTVD_FLAG_NO_CUDA_GRAPH))):
        model, _ = _build_model(W.DEFAULT_ENC_CONFIG, W.DEFAULT_DEC_CONFIG, full_sd, "bf16", engine_max_batch=B, engine_max_beams=K, **kw)
        runs = [_call(model, b, **gk)[0].cpu() for _ in range(2)]
        assert runs[0].shape == (B * K, 18)
        assert torch.equal(runs[0], runs[1]), f"{name}: repeated calls differ"
        outs[name] = runs[0]
        del model
        torch.cuda.empty_cache()
    assert torch.equal(outs["separate_calls"], outs["whole_round"]), "whole-round graph differs from separate calls"
    assert torch.equal(outs["no_cuda_graph"], outs["whole_round"]), "eager decode differs from the captured graph"

    e = _engine(enc_cfg, dec_cfg, full_sd, "bf16", b)
    try:
        # one group pays nothing for the groups machinery: the penalty only acts on groups after the first, so with G = 1 it
        # changes no id, no score and no launch
        res = []
        for penalty in (0.0, 0.7):
            l0 = e.launch_count
            out, sc = e.generate(B, num_beams=K, num_beam_groups=1, diversity_penalty=penalty, num_return_sequences=K, ngram_blocking_size=4,
                                 want_scores=True, **_hist(b))
            res.append((out.cpu(), sc.cpu(), e.launch_count - l0))
        assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1]) and res[0][2] == res[1][2], (res[0][2], res[1][2])
        grouped = e.generate(B, num_beams=K, num_beam_groups=3, diversity_penalty=0.5, num_return_sequences=K, ngram_blocking_size=4,
                             **_hist(b)).cpu()
        assert torch.equal(grouped, outs["separate_calls"])
        # the penalty takes effect: G = K beams of one token each are pairwise distinct with a large penalty, identical without
        apart = e.generate(B, num_beams=K, num_beam_groups=K, diversity_penalty=1e4, num_return_sequences=K).cpu().view(B, K, 18)
        same = e.generate(B, num_beams=K, num_beam_groups=K, diversity_penalty=0.0, num_return_sequences=K).cpu().view(B, K, 18)
        distinct = sum(len({tuple(r) for r in apart[i].tolist()}) == K for i in range(B))
        identical = sum(len({tuple(r) for r in same[i].tolist()}) == 1 for i in range(B))
        print(f"bf16 B = {B}, G = K = {K}: images with pairwise distinct beams at penalty 1e4: {distinct} of {B}; "
              f"with identical beams at penalty 0: {identical} of {B}")
        assert distinct == B and identical == B
    finally:
        e.close()


# ---- GPU: dialog loop and CLI ---------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_dialog_with_beam_groups(tiny_cfgs, tiny_sd):
    from gst_visdial_b200 import weights as W
    from gst_visdial_b200.dialog import generate_dialogs
    from test_gpu_model import _build_model
    enc_cfg, _ = tiny_cfgs
    B, rounds, K = 3, 2, 4
    b = history_batch(enc_cfg, 0, B, rounds=1)
    q_model, _ = _build_model(W.TINY_ENC_CONFIG, W.TINY_DEC_CONFIG, tiny_sd, "fp32", model="enc_dec_q", engine_max_beams=K)
    a_model, _ = _build_model(W.TINY_ENC_CONFIG, W.TINY_DEC_CONFIG, tiny_sd, "fp32", model="enc_dec_a", engine_max_beams=K)
    q_kwargs = dict(num_beams=K, num_beam_groups=2, diversity_penalty=0.5, ngram_blocking_size=4, **_GREEDY)
    a_kwargs = dict(num_beams=K, num_beam_groups=K, diversity_penalty=1.0, ngram_blocking_size=0, **_GREEDY)
    res = generate_dialogs(a_model, b, q_model=q_model, num_rounds=rounds, q_kwargs=q_kwargs, a_kwargs=a_kwargs, with_ppl=True,
                           device="cuda:0", answer_candidates=K)
    assert res.questions.shape == (B, rounds, 18) and res.answers.shape == (B, rounds, 18)
    assert torch.isfinite(res.answer_ppl).all()
    for r in range(rounds):
        q = res.questions[:, r].cpu()
        assert ((q == R.EOS).sum(1) <= 1).all() and (q[:, 0] != 0).all()
        assert (res.answers[:, r].cpu()[:, 0] != 0).any()


@pytest.mark.gpu
def test_generate_cli_beam_groups(tmp_path):
    import json
    import subprocess
    import sys
    from helpers import ROOT
    cmd = [sys.executable, os.path.join(ROOT, "generate.py"), "-synthetic", "8", "-batch_size", "8", "-num_beams", "6", "-num_beam_groups", "3",
           "-diversity_penalty", "0.5", "-answer_candidates", "3", "-q_num_beams", "4", "-q_num_beam_groups", "2", "-q_diversity_penalty", "0.5",
           "-num_rounds", "2", "-save_path", str(tmp_path), "-save_name", "o.json"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout + r.stderr
    out = json.load(open(tmp_path / "o.json"))
    assert len(out) == 8 and all(len(d["dialog"]) == 2 for d in out)


# ---- GPU: argument checks ------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_group_rejections(tiny_cfgs, tiny_sd):
    from gst_visdial_b200 import weights as W
    from gst_visdial_b200._lib import GstvdError
    from test_gpu_model import _build_model, _call
    GSTVD_ERR_INVALID = -1
    enc_cfg, dec_cfg = tiny_cfgs
    B = 2
    b = history_batch(enc_cfg, 0, B)
    rnd = (b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"], b["enc_image_mask"])
    bad = [dict(num_beams=6, num_beam_groups=4), dict(num_beams=4, num_beam_groups=0), dict(num_beams=1, num_beam_groups=2),
           dict(num_beams=4, num_beam_groups=2, diversity_penalty=-0.5), dict(num_beams=4, num_beam_groups=2, diversity_penalty=float("nan")),
           dict(num_beams=4, num_beam_groups=2, diversity_penalty=float("inf")), dict(num_beams=4, diversity_penalty=-1.0)]
    e = _engine(enc_cfg, dec_cfg, tiny_sd, "fp32", b)
    try:
        for kw in bad:
            with pytest.raises(GstvdError) as ei:
                e.generate(B, **kw)
            assert ei.value.status == GSTVD_ERR_INVALID, kw
            with pytest.raises(GstvdError) as ei:
                e.round(*rnd, **kw)
            assert ei.value.status == GSTVD_ERR_INVALID, kw
        assert e.generate(B, num_beams=6, num_beam_groups=6, diversity_penalty=2.0, num_return_sequences=6).shape == (B * 6, 18)
    finally:
        e.close()
    model, _ = _build_model(W.TINY_ENC_CONFIG, W.TINY_DEC_CONFIG, tiny_sd, "fp32", engine_max_beams=6)
    with pytest.raises(ValueError):
        _call(model, b, num_beams=1, num_beam_groups=2, ngram_blocking_size=0, **_GREEDY)
    for kw in bad:
        if kw["num_beams"] > 1:
            with pytest.raises(GstvdError):
                _call(model, b, ngram_blocking_size=0, **kw, **_GREEDY)
