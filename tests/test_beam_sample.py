"""Beam sampling: num_beams > 1 with do_sample (HF 4.16.2 beam_sample; include/gstvd.h GSTVD_SELECT_BEAM_SAMPLE, contract in
oracle/beam_sample.py).

CPU: the oracle's Gumbel-top-2K draw has the law of sequential sampling without replacement (chi-square against the enumerated
Plackett-Luce set probabilities); structural properties of the oracle (all beams start at 0, 2K distinct finite entries per draw, nothing
outside top-k' / the nucleus and nothing banned is drawn, the temperature compounds through the beam scores); the RNG mirror and the
independence of an image's draws from the row_offset split; the CLI flags.
GPU: ids identical to the oracle (scores within 1e-4) in fp32 on every call path for K = 2, 3, 4, N = 1, 2, with and without blocking
and a decoder prefix, at tiny and full size; search n equals an N = 1 call seeded candidate_seed(seed, n) and a row_offset split changes
nothing; the bf16 product path agrees across call paths, is reproducible per seed and never emits a banned n-gram; the dialog loop and
generate.py run with beam sampling; every rejected argument raises.
"""
import ctypes
import itertools
import os

import numpy as np
import pytest
import torch

from helpers import R, history_batch
from oracle import beam as OB
from oracle import beam_ngram as BN
from oracle import beam_sample as BS
from test_beam_ngram import FULL_TOKS, TINY_TOKS, _boosted, _hits
from test_beam_ngram import _with_question as _with_de_bruijn
from test_candidates import _sub
from test_decoder_prefix import _prefixes

_WARP = dict(temperature=0.7, top_k=7, top_p=0.0)


def _random_logits(rows, V, T, seed, eos_from=3):
    g = torch.Generator().manual_seed(seed)
    logits = [torch.randn(rows, V, generator=g) * 3 for _ in range(T)]
    for lg in logits[eos_from:]:
        lg[:, OB.EOS] += 3.0
    return logits


# ---- CPU: the draw -------------------------------------------------------------------------------------------------
def test_gumbel_top_2k_has_the_law_of_sampling_without_replacement():
    from scipy.stats import chi2
    K, V, draws = 2, 5, 40000
    w = np.array([0.3, -0.2, 1.1, -1.5, 0.0, 0.8, -0.7, 0.4, -2.2, 0.1], dtype=np.float32)   # the K*V warped scores of one search
    p = np.exp(w.astype(np.float64) - w.max())
    p /= p.sum()
    exact = {}
    for perm in itertools.permutations(range(K * V), 2 * K):              # Plackett-Luce: sequential draws without replacement
        pr, left = 1.0, 1.0
        for i in perm:
            pr *= p[i] / left
            left -= p[i]
        key = frozenset(perm)
        exact[key] = exact.get(key, 0.0) + pr
    assert abs(sum(exact.values()) - 1.0) < 1e-12
    counts = {}
    flat = np.arange(K * V)
    for seed in range(draws):
        keys = BS.gumbel_keys(w, BS.uniforms(BS.candidate_seed(seed, 0), 0, 0, flat))
        drawn = frozenset(np.argsort(-keys, kind="stable")[: 2 * K].tolist())
        counts[drawn] = counts.get(drawn, 0) + 1
    obs, exp, pool_o, pool_e = [], [], 0, 0.0
    for key, pe in exact.items():
        if pe * draws >= 5:
            obs.append(counts.get(key, 0)); exp.append(pe * draws)
        else:
            pool_o += counts.get(key, 0); pool_e += pe * draws
    obs.append(pool_o); exp.append(pool_e)
    stat = sum((o - e) ** 2 / e for o, e in zip(obs, exp))
    pval = chi2.sf(stat, len(obs) - 1)
    assert pval > 1e-3, (stat, len(obs), pval)


def test_rng_mirror():
    from gst_visdial_b200.models.visual_dialog_model import _splitmix64, candidate_seed
    for x in (0, 1, 2**63 + 5, 2**64 - 1):
        assert int(BS.splitmix64(np.array([x], dtype=np.uint64))[0]) == _splitmix64(x)
    for s in (0, 9, 2**64 - 3):
        assert all(BS.candidate_seed(s, n) == candidate_seed(s, n) for n in range(8))
    # u = ((h >> 11) + 0.5) 2^-53 with h = splitmix64(splitmix64(sd ^ splitmix64((grow << 20) ^ t)) ^ flat), in plain Python integers
    sd, grow, t, flat = 0x1234567890ABCDEF, 77, 5, np.array([3, 40000, 3])
    h = [_splitmix64(_splitmix64(sd ^ _splitmix64(((grow << 20) & BS.M64) ^ t)) ^ int(f)) for f in flat]
    u = BS.uniforms(sd, grow, t, flat)
    assert u.tolist() == [((x >> 11) + 0.5) * 2.0 ** -53 for x in h]
    assert u[0] == u[2] and u[0] != u[1] and ((0 < u) & (u < 1)).all()
    assert BS.uniforms(sd, grow, t + 1, flat)[0] != u[0] and BS.uniforms(sd, grow + 1, t, flat)[0] != u[0]


# ---- CPU: oracle structure -----------------------------------------------------------------------------------------
_HIST_TOKS = (120, 121)


def _hist():
    a, c = _HIST_TOKS
    return [[R.CLS, a, c, a, a, c, c, a, c, R.EOS], [0, 130, a, a, c, a, 131, 0], [a, c, a, c, c]]


@pytest.mark.parametrize("top_p", [0.0, 0.6])
def test_beam_sample_oracle_structure(top_p):
    B, N, K, V, T, n = 3, 2, 3, 160, 10, 2
    temp, top_k = 0.7, 5
    logits = _random_logits(B * N * K, V, T, seed=4)
    for lg in logits:
        lg[:, list(_HIST_TOKS)] += 3.0                                    # the history bigrams compete: blocking has work to do
    hist = _hist()
    st = BS.BeamSampleState(B, K, V, T, N=N, temperature=temp, top_k=top_k, top_p=top_p, seed=11)
    assert (st.beam_scores == 0).all(), "beam_sample starts every beam at 0"
    checked = 0
    for t, lg in enumerate(logits):
        if bool(st.done.all()):
            break
        prev_scores = st.beam_scores.clone()
        banned = st.banned(hist, n)
        was_done = st.done.clone()
        idx, tok, sc = st.step(lg, ngram_blocking_size=n, hist=hist)
        w, lid, kept = st.last_lists
        lp = lg - OB.log_z(lg)
        for s in range(st.B):
            if was_done[s]:
                assert (tok[s] == R.PAD).all() and (sc[s] == 0).all() and (idx[s] == 0).all()
                continue
            draw = st.last_draw[s]
            assert len(draw) == 2 * K and len(set(draw)) == 2 * K
            for c in draw:
                k, j = divmod(c, BS.NSEL)
                wv, w_tok = w[s, k, j], int(lid[s, k, j])
                assert torch.isfinite(wv)
                assert j < int(kept[s, k]), "drawn outside the top-k' / nucleus set"
                assert w_tok not in banned[s * K + k], "drew a banned token"
                # the temperature compounds: w = fp32(fp32(fp32(x - logZ) + beam_score) / T), beam_score itself a warped value
                want = ((lp[s * K + k, w_tok] + prev_scores[s, k]) / torch.tensor(temp)).float()
                assert wv == want
                checked += 1
            for k in range(K):
                kk = int(kept[s, k])
                assert 2 <= kk
                row = w[s, k]
                assert kk <= BS.NSEL and (row[kk - 1] >= row[max(top_k, 2) - 1] or kk <= max(top_k, 2))
                if top_p == 0.0:
                    assert kk == int((row >= row[max(top_k, 2) - 1]).sum())
                else:
                    p = torch.softmax(row[: int((row >= row[max(top_k, 2) - 1]).sum())].double(), 0)
                    if kk > 2:
                        assert float(p[: kk - 1].sum()) <= top_p + 1e-6, "a kept rank came after the nucleus was full"
                    if kk < len(p):
                        assert float(p[:kk].sum()) > top_p - 1e-6, "the nucleus stopped early"
        if t >= 1:
            # the new beam scores are drawn warped values: a surviving beam's score divided by T is folded into the next step
            assert not torch.equal(st.beam_scores, prev_scores)
    assert checked > 100


def test_beam_sample_oracle_row_offset_split():
    B, N, K, V, T = 4, 2, 2, 120, 8
    logits = _random_logits(B * N * K, V, T, seed=8)
    kw = dict(temperature=0.7, top_k=7, top_p=0.9, seed=123)
    whole = BS.BeamSampleState(B, K, V, T, N=N, **kw)
    parts = [BS.BeamSampleState(2, K, V, T, N=N, row_offset=lo, **kw) for lo in (0, 2)]
    rows = 2 * N * K
    for lg in logits:
        whole.step(lg)
        for i, st in enumerate(parts):
            st.step(lg[i * rows: (i + 1) * rows])
    seq, sc = whole.finalize()
    got = [st.finalize() for st in parts]
    assert torch.equal(seq, torch.cat([g[0] for g in got])) and torch.equal(sc, torch.cat([g[1] for g in got]))
    other = BS.BeamSampleState(B, K, V, T, N=N, **dict(kw, seed=124))
    for lg in logits:
        other.step(lg)
    assert not torch.equal(other.finalize()[0], seq), "a different seed draws something else"


def test_beam_sample_oracle_search_is_a_seeded_single_search():
    B, N, K, V, T = 2, 3, 2, 120, 7
    logits = _random_logits(B * N * K, V, T, seed=5)
    multi = BS.BeamSampleState(B, K, V, T, N=N, seed=9)
    singles = [BS.BeamSampleState(B, K, V, T, N=1, seed=BS.candidate_seed(9, n)) for n in range(N)]
    for lg in logits:
        multi.step(lg)
        per = lg.view(B, N, K, V)
        for n, st in enumerate(singles):
            st.step(per[:, n].reshape(B * K, V))
    seq = multi.finalize()[0].view(B, N, T)
    for n, st in enumerate(singles):
        assert torch.equal(seq[:, n], st.finalize()[0])


def test_beam_sample_oracle_rejects_bad_args():
    for kw in (dict(K=1), dict(K=9), dict(N=0), dict(temperature=0.0), dict(temperature=float("inf")), dict(temperature=float("nan")),
               dict(top_p=-0.1), dict(top_p=1.5), dict(top_k=0), dict(top_k=17)):
        args = dict(K=3, N=1, temperature=0.7, top_k=7, top_p=0.0)
        args.update(kw)
        with pytest.raises(ValueError):
            BS.BeamSampleState(1, args["K"], 50, 5, N=args["N"], temperature=args["temperature"], top_k=args["top_k"], top_p=args["top_p"])


def test_beam_sample_options(tmp_path):
    from gst_visdial_b200 import options
    base = ["-save_path", str(tmp_path)]
    p = options.read_command_line(base)
    assert (p["beam_sample"], p["q_beam_sample"]) == (False, False)
    p = options.read_command_line(base + ["-num_beams", "4", "-beam_sample", "-answer_candidates", "2", "-q_num_beams", "3", "-q_beam_sample"])
    assert (p["beam_sample"], p["q_beam_sample"], p["engine_max_beams"]) == (True, True, 8)
    p = options.read_command_line(base + ["-num_beams", "4", "-answer_candidates", "2"])
    assert p["engine_max_beams"] == 4, "beam search returns the N best of its K beams: no extra rows"
    for bad in (["-beam_sample"], ["-num_beams", "1", "-beam_sample"], ["-q_beam_sample"], ["-q_num_beams", "1", "-q_beam_sample"],
                ["-num_beams", "4", "-num_beam_groups", "2", "-beam_sample"],
                ["-q_num_beams", "4", "-q_num_beam_groups", "2", "-q_beam_sample"],
                ["-num_beams", "3", "-answer_candidates", "3", "-beam_sample"]):
        with pytest.raises(SystemExit):
            options.read_command_line(base + bad)


# ---- GPU: fp32 against the oracle ----------------------------------------------------------------------------------
_ORACLE = {}
_SEED = 0x5EED


def _oracle(sd, enc_cfg, dec_cfg, b, K, N, n, prefix=None, tag="", seed=_SEED, warp=_WARP):
    key = (tag, K, N, n, prefix is not None, seed, tuple(sorted(warp.items())))
    if key not in _ORACLE:
        with torch.no_grad():
            _ORACLE[key] = BS.beam_sample(sd, enc_cfg, dec_cfg, b, K, N, seed=seed, ngram_blocking_size=n, prefix=prefix, **warp)
    return _ORACLE[key]


def _hist_kw(b):
    return dict(hist_ids=b["enc_input_ids"], hist_segments=b["enc_segments"])


def _path_kw(path):
    from gst_visdial_b200 import _lib
    return {"separate_calls": dict(engine_round_graph=False), "whole_round": {},
            "no_cuda_graph": dict(engine_flags=_lib.GSTVD_FLAG_NO_CUDA_GRAPH)}[path]


def _engine(enc_cfg, dec_cfg, sd, dtype, b, **kw):
    from gst_visdial_b200.engine import Engine
    B = b["enc_input_ids"].shape[0]
    kw.setdefault("max_beams", 8)
    e = Engine(enc_cfg, dec_cfg, dtype=dtype, max_batch=B, **kw)
    e.load_state_dict(sd)
    o = e.encode(b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"], b["enc_image_mask"])
    e.prefill_cross(B, o["Le"])
    return e


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["separate_calls", "whole_round", "no_cuda_graph"])
@pytest.mark.parametrize("top_p", [0.0, 0.6])
@pytest.mark.parametrize("n", [0, 4])
@pytest.mark.parametrize("N", [1, 2])
@pytest.mark.parametrize("K", [2, 3, 4])
def test_tiny_fp32_beam_sample_matches_oracle(tiny_cfgs, tiny_sd, K, N, n, top_p, path):
    from gst_visdial_b200 import weights as W
    from test_gpu_model import _build_model, _call
    enc_cfg, dec_cfg = tiny_cfgs
    sd = _boosted(tiny_sd, TINY_TOKS)
    sd["decoder.decoder.lm_head.bias"][R.EOS] += 5.0             # hypotheses end early and compete for the heap
    b = _with_de_bruijn(history_batch(enc_cfg, 0, 3), TINY_TOKS)
    warp = dict(_WARP, top_p=top_p)                              # top_p > 0: the kernel's nucleus cut against oracle.kept_count
    ref, ref_sc = _oracle(sd, enc_cfg, dec_cfg, b, K, N, n, tag="tiny", warp=warp)
    if n:
        assert not any(_hits(b, ref[::N], 4))
    model, _ = _build_model(W.TINY_ENC_CONFIG, W.TINY_DEC_CONFIG, sd, "fp32", engine_max_beams=8, **_path_kw(path))
    eng = model.module._engine(torch.device("cuda:0"))
    gk = dict(num_beams=K, do_sample=True, ngram_blocking_size=n, num_return_sequences=N, seed=_SEED, **warp)
    seq, _ = _call(model, b, **gk)
    assert torch.equal(seq.cpu(), ref), f"{seq.cpu().tolist()} vs {ref.tolist()}"
    seq2, sc2 = eng.generate(3, want_scores=True, **gk, **_hist_kw(b))
    assert torch.equal(seq2.cpu(), ref)
    assert torch.allclose(sc2.cpu().double(), ref_sc, atol=1e-4), (sc2, ref_sc)


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["separate_calls", "whole_round", "no_cuda_graph"])
def test_tiny_fp32_beam_sample_from_prefix_matches_oracle(tiny_cfgs, tiny_sd, path):
    from gst_visdial_b200 import weights as W
    from test_gpu_model import _build_model, _call
    enc_cfg, dec_cfg = tiny_cfgs
    K, N, n = 3, 2, 4
    sd = _boosted(tiny_sd, TINY_TOKS)
    b = _with_de_bruijn(history_batch(enc_cfg, 0, 3), TINY_TOKS)
    pre = _prefixes(3, 5, enc_cfg.vocab_size)
    pre[0, -3:] = torch.tensor([TINY_TOKS[0]] * 3)                 # the first step's key lies in the prefix
    ref, ref_sc = _oracle(sd, enc_cfg, dec_cfg, b, K, N, n, prefix=pre, tag="tiny")
    model, _ = _build_model(W.TINY_ENC_CONFIG, W.TINY_DEC_CONFIG, sd, "fp32", engine_max_beams=8, **_path_kw(path))
    eng = model.module._engine(torch.device("cuda:0"))
    gk = dict(num_beams=K, do_sample=True, ngram_blocking_size=n, num_return_sequences=N, seed=_SEED, **_WARP)
    seq, dec = _call(model, b, dec_ids=pre.clone(), **gk)
    assert torch.equal(seq.cpu(), ref), f"{seq.cpu().tolist()} vs {ref.tolist()}"
    assert torch.equal(dec.cpu(), pre)
    seq2, sc2 = eng.generate(3, want_scores=True, prefix=pre, **gk, **_hist_kw(b))
    assert torch.equal(seq2.cpu(), ref)
    assert torch.allclose(sc2.cpu().double(), ref_sc, atol=1e-4), (sc2, ref_sc)


@pytest.mark.gpu
def test_full_fp32_beam_sample_matches_oracle(full_cfgs, full_sd):
    enc_cfg, dec_cfg = full_cfgs
    K, N, n = 3, 2, 4
    sd = _boosted(full_sd, FULL_TOKS)
    b = _with_de_bruijn(history_batch(enc_cfg, 0, 2), FULL_TOKS)
    ref, ref_sc = _oracle(sd, enc_cfg, dec_cfg, b, K, N, n, tag="full")
    e = _engine(enc_cfg, dec_cfg, sd, "fp32", b)
    try:
        seq, sc = e.generate(2, num_beams=K, do_sample=True, ngram_blocking_size=n, want_scores=True, num_return_sequences=N, seed=_SEED,
                             **_WARP, **_hist_kw(b))
        assert torch.equal(seq.cpu(), ref), f"{seq.cpu().tolist()} vs {ref.tolist()}"
        assert torch.allclose(sc.cpu().double(), ref_sc, atol=1e-4)
    finally:
        e.close()


@pytest.mark.gpu
def test_tiny_fp32_searches_are_seeded_single_calls(tiny_cfgs, tiny_sd):
    from gst_visdial_b200.models.visual_dialog_model import candidate_seed
    enc_cfg, dec_cfg = tiny_cfgs
    B, K, N, seed = 4, 2, 4, 91
    b = _with_de_bruijn(history_batch(enc_cfg, 0, B), TINY_TOKS)
    e = _engine(enc_cfg, dec_cfg, tiny_sd, "fp32", b)
    try:
        kw = dict(num_beams=K, do_sample=True, ngram_blocking_size=4, **_WARP, **_hist_kw(b))
        multi, msc = e.generate(B, seed=seed, num_return_sequences=N, want_scores=True, **kw)
        multi, msc = multi.cpu().view(B, N, 18), msc.cpu().view(B, N)
        for n in range(N):
            one, osc = e.generate(B, seed=candidate_seed(seed, n), want_scores=True, **kw)
            assert torch.equal(multi[:, n], one.cpu()), n
            assert torch.equal(msc[:, n], osc.cpu()), n
        assert len({tuple(multi[i, n].tolist()) for i in range(B) for n in range(N)}) > B, "the searches all drew the same"
    finally:
        e.close()
    parts = []
    for lo, hi in ((0, 1), (1, B)):
        sub = _sub(b, lo, hi)
        e = _engine(enc_cfg, dec_cfg, tiny_sd, "fp32", sub)
        try:
            parts.append(e.generate(hi - lo, seed=seed, num_return_sequences=N, row_offset=lo, num_beams=K, do_sample=True,
                                    ngram_blocking_size=4, **_WARP, **_hist_kw(sub)).cpu())
        finally:
            e.close()
    assert torch.equal(torch.cat(parts).view(B, N, 18), multi)


# ---- GPU: bf16 product path ----------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_full_bf16_beam_sample(full_cfgs, full_sd):
    from gst_visdial_b200 import _lib, weights as W
    from gst_visdial_b200.models.visual_dialog_model import candidate_seed
    from test_gpu_model import _build_model, _call
    enc_cfg, dec_cfg = full_cfgs
    B, K, N, seed = 64, 4, 2, 2024
    b = history_batch(enc_cfg, 0, B)
    gk = dict(num_beams=K, do_sample=True, ngram_blocking_size=4, num_return_sequences=N, seed=seed, **_WARP)
    outs = {}
    for name, kw in (("whole_round", {}), ("separate_calls", dict(engine_round_graph=False)),
                     ("no_cuda_graph", dict(engine_round_graph=False, engine_flags=_lib.GSTVD_FLAG_NO_CUDA_GRAPH))):
        model, _ = _build_model(W.DEFAULT_ENC_CONFIG, W.DEFAULT_DEC_CONFIG, full_sd, "bf16", engine_max_batch=B, engine_max_beams=N * K, **kw)
        runs = [_call(model, b, **gk)[0].cpu() for _ in range(2)]
        assert runs[0].shape == (B * N, 18)
        assert torch.equal(runs[0], runs[1]), f"{name}: the same seed gave different ids"
        outs[name] = runs[0]
        if name == "whole_round":
            other = _call(model, b, **dict(gk, seed=seed + 1))[0].cpu()
            assert not torch.equal(other, runs[0]), "a different seed gave the same ids"
        del model
        torch.cuda.empty_cache()
    assert torch.equal(outs["separate_calls"], outs["whole_round"]), "whole-round graph differs from separate calls"
    assert torch.equal(outs["no_cuda_graph"], outs["whole_round"]), "eager decode differs from the captured graph"
    hist = BN.question_history(b["enc_input_ids"], b["enc_segments"])
    seq = outs["whole_round"]
    assert not any(BN.contains_banned_ngram(hist[r // N], seq[r].tolist(), 4) for r in range(B * N)), "a banned 4-gram was emitted"
    assert (seq[:, 0] != 0).all()

    e = _engine(enc_cfg, dec_cfg, full_sd, "bf16", b)
    try:
        kw = dict(num_beams=K, do_sample=True, ngram_blocking_size=4, **_WARP, **_hist_kw(b))
        multi = e.generate(B, seed=seed, num_return_sequences=N, **kw).cpu().view(B, N, 18)
        assert torch.equal(multi.view(B * N, 18), outs["separate_calls"])
        same = torch.stack([(multi[:, n] == e.generate(B, seed=candidate_seed(seed, n), **kw).cpu()).all(1) for n in range(N)], 1)
        # bf16: N * K = 8 rows per image against K = 4 in the single call run different GEMM tilings, so a near tie may tip
        # (measured on an NVIDIA B200: 128 of 128 equal)
        print(f"bf16 B = {B}, K = {K}, N = {N}: searches equal to their N = 1 call: {int(same.sum())} of {B * N}")
        assert same.float().mean() > 0.5
    finally:
        e.close()


# ---- GPU: dialog loop and CLI ---------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_dialog_with_beam_sampling(tiny_cfgs, tiny_sd):
    from gst_visdial_b200 import weights as W
    from gst_visdial_b200.dialog import generate_dialogs
    from test_gpu_model import _build_model
    enc_cfg, _ = tiny_cfgs
    B, rounds, K, N = 3, 2, 4, 2
    b = history_batch(enc_cfg, 0, B, rounds=1)
    q_model, _ = _build_model(W.TINY_ENC_CONFIG, W.TINY_DEC_CONFIG, tiny_sd, "fp32", model="enc_dec_q", engine_max_beams=K)
    a_model, _ = _build_model(W.TINY_ENC_CONFIG, W.TINY_DEC_CONFIG, tiny_sd, "fp32", model="enc_dec_a", engine_max_beams=N * K)
    q_kwargs = dict(num_beams=K, do_sample=True, ngram_blocking_size=4, **_WARP)
    a_kwargs = dict(num_beams=K, do_sample=True, ngram_blocking_size=0, **_WARP)
    res = generate_dialogs(a_model, b, q_model=q_model, num_rounds=rounds, q_kwargs=q_kwargs, a_kwargs=a_kwargs, with_ppl=True,
                           device="cuda:0", answer_candidates=N)
    assert res.questions.shape == (B, rounds, 18) and res.answers.shape == (B, rounds, 18)
    assert torch.isfinite(res.answer_ppl).all()
    for r in range(rounds):
        q = res.questions[:, r].cpu()
        assert ((q == R.EOS).sum(1) <= 1).all() and (q[:, 0] != 0).all()
        assert (res.answers[:, r].cpu()[:, 0] != 0).any()


@pytest.mark.gpu
def test_generate_cli_beam_sample(tmp_path):
    import json
    import subprocess
    import sys
    from helpers import ROOT
    cmd = [sys.executable, os.path.join(ROOT, "generate.py"), "-synthetic", "8", "-batch_size", "8", "-num_beams", "4", "-beam_sample",
           "-answer_candidates", "2", "-q_num_beams", "3", "-q_beam_sample", "-num_rounds", "2", "-save_path", str(tmp_path),
           "-save_name", "o.json"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout + r.stderr
    out = json.load(open(tmp_path / "o.json"))
    assert len(out) == 8 and all(len(d["dialog"]) == 2 for d in out)


# ---- GPU: argument checks ------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_beam_sample_rejections(tiny_cfgs, tiny_sd):
    from gst_visdial_b200 import _lib, weights as W
    from gst_visdial_b200._lib import GstvdError
    from test_gpu_model import _build_model, _call
    INVALID, UNSUPPORTED = -1, -3
    enc_cfg, dec_cfg = tiny_cfgs
    B = 2
    b = history_batch(enc_cfg, 0, B)
    rnd = (b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"], b["enc_image_mask"])
    ok = dict(num_beams=3, do_sample=True, **_WARP)
    bad = [(dict(num_beams=9), INVALID), (dict(num_return_sequences=0), INVALID), (dict(num_return_sequences=3), INVALID),
           (dict(num_beams=4, num_beam_groups=2), INVALID), (dict(temperature=0.0), INVALID), (dict(temperature=-1.0), INVALID),
           (dict(temperature=float("inf")), INVALID), (dict(temperature=float("nan")), INVALID), (dict(top_p=-0.5), INVALID),
           (dict(top_p=1.5), INVALID), (dict(top_p=float("nan")), INVALID), (dict(top_k=0), UNSUPPORTED), (dict(top_k=17), UNSUPPORTED)]
    e = _engine(enc_cfg, dec_cfg, tiny_sd, "fp32", b)
    try:
        for kw, status in bad:
            args = dict(ok, **kw)
            with pytest.raises(GstvdError) as ei:
                e.generate(B, **args)
            assert ei.value.status == status, kw
            with pytest.raises(GstvdError) as ei:
                e.round(*rnd, **args)
            assert ei.value.status == status, kw
        # num_beams < 2 in beam-sampling mode: Engine maps num_beams = 1 to the sampler, so call the C ABI with mode 2 directly
        gp = _lib.GstvdGenParams()
        gp.mode, gp.num_beams, gp.max_new_tokens, gp.top_k, gp.temperature = _lib.GSTVD_SELECT_BEAM_SAMPLE, 1, 18, 7, 0.7
        gp.num_return_sequences = gp.num_beam_groups = 1
        out = torch.empty(B, 18, dtype=torch.int64, device="cuda:0")
        for call in ("generate", "round"):
            if call == "generate":
                rc = e.lib.gstvd_generate(e.ctx, B, ctypes.byref(gp), None, 1, None, None, 0, ctypes.c_void_p(out.data_ptr()), None,
                                          e._stream())
            else:
                ids, seg = (t.cuda().long().contiguous() for t in (rnd[0], rnd[3]))
                feat, loc, att, imask = (t.cuda().float().contiguous() for t in (rnd[1], rnd[2], rnd[4], rnd[5]))
                rc = e.lib.gstvd_round(e.ctx, B, ids.shape[1], feat.shape[1], *[ctypes.c_void_p(t.data_ptr()) for t in
                                       (ids, seg, att, feat, loc, imask)], ctypes.byref(gp), None, 1,
                                       ctypes.c_void_p(out.data_ptr()), None, e._stream())
            assert rc == INVALID, (call, rc)
        assert e.generate(B, num_return_sequences=2, **dict(ok, num_beams=4)).shape == (B * 2, 18)
        assert e.generate(B, num_beams=2, do_sample=True, **dict(_WARP, top_k=1, top_p=1.0)).shape == (B, 18)
    finally:
        e.close()
    model, _ = _build_model(W.TINY_ENC_CONFIG, W.TINY_DEC_CONFIG, tiny_sd, "fp32", engine_max_beams=8)
    with pytest.raises(ValueError):
        _call(model, b, num_beams=4, num_beam_groups=2, do_sample=True, ngram_blocking_size=0, **_WARP)
    with pytest.raises(GstvdError):
        _call(model, b, num_beams=3, do_sample=True, num_return_sequences=3, ngram_blocking_size=0, **_WARP)
