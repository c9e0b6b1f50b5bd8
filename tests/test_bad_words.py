"""HF bad_words_ids in every decode mode (include/gstvd.h gstvd_generate, CPU oracle oracle/decode_args.py, pinned on the installed
transformers by oracle/gen_golden_bad_words.py)."""
import ctypes
import json
import os

import numpy as np
import pytest
import torch

from helpers import ROOT, R, history_batch
from oracle import decode_args as DA
from oracle import processors as LP
from oracle.beam_nbest import finalize_nbest
from test_decoder_prefix import A4, _prefixes, _with_bias, _with_question

GOLDEN = os.path.join(ROOT, "tests", "golden", "bad_words.npz")


# ---- CPU: the restatement -------------------------------------------------------------------------------------------
def _words(flat):
    out, cur = [], []
    for w in flat.tolist():
        if w == -1:
            out.append(cur); cur = []
        else:
            cur.append(w)
    return out


def test_restatement_equals_goldens():
    g = np.load(GOLDEN)
    names = sorted({k.rsplit("_", 1)[0] for k in g.files})
    assert len(names) >= 8
    for n in names:
        ids = g[f"{n}_ids"].tolist()
        out = DA.apply_bad_words(torch.from_numpy(g[f"{n}_scores"]), ids, _words(g[f"{n}_words"]))
        assert torch.equal(out, torch.from_numpy(g[f"{n}_out"])), n


def test_restatement_equals_installed_hf_but_where_4_16_2_differs():
    pytest.importorskip("transformers")
    from oracle.gen_golden_bad_words import cases, hf_apply
    for name, s, ids, words in cases():
        ours, hf = DA.apply_bad_words(s, ids.tolist(), words), hf_apply(s, ids, words)
        extra = [(r, w[-1]) for r in range(ids.shape[0]) for w in words
                 if w != [R.EOS] and len(w) - 1 == ids.shape[1] and ids[r].tolist() == w[:-1]]
        expect = hf.clone()
        for r, w in extra:
            expect[r, w] = -float("inf")
        assert torch.equal(ours, expect), name


def test_rule_examples():
    d = [101, 5, 6, 7]
    assert DA.bad_words_banned(d, [[9]]) == [9]                            # one id: always
    assert DA.bad_words_banned(d, [[6, 7, 8]]) == [8]                      # the tail matches
    assert DA.bad_words_banned(d, [[5, 7, 8]]) == []
    assert DA.bad_words_banned(d, [[101, 5, 6, 7, 3]]) == [3]              # L - 1 == cur_len: 4.16.2 tests it
    assert DA.bad_words_banned(d, [[1, 101, 5, 6, 7, 3]]) == []            # longer than d + 1
    assert DA.bad_words_banned(d, [[102]]) == []                            # [SEP] alone is dropped
    assert DA.bad_words_banned(d, [[7, 102]]) == [102]                      # a longer sequence may end in [SEP]
    assert DA.completes_bad_word([101, 5], [6, 7, 102], [[5, 6, 7]]) and not DA.completes_bad_word([101], [5, 6], [[5, 7]])


def test_cli_flags(tmp_path):
    from gst_visdial_b200 import options
    base = ["-save_path", str(tmp_path)]
    p = options.read_command_line(base)
    assert (p["length_penalty"], p["early_stopping"], p["bad_words_ids"]) == (1.0, False, None)
    assert (p["q_length_penalty"], p["q_early_stopping"], p["q_bad_words_ids"]) == (1.0, False, None)
    f = tmp_path / "bw.json"
    f.write_text(json.dumps([[100], [2054, 2064]]))
    p = options.read_command_line(base + ["-length_penalty", "1.5", "-early_stopping", "-bad_words_ids", str(f), "-q_length_penalty", "-0.5",
                                          "-q_early_stopping", "-q_bad_words_ids", str(f)])
    assert (p["length_penalty"], p["early_stopping"], p["bad_words_ids"]) == (1.5, True, [[100], [2054, 2064]])
    assert (p["q_length_penalty"], p["q_early_stopping"], p["q_bad_words_ids"]) == (-0.5, True, [[100], [2054, 2064]])
    bad_files = {"empty_seq": [[1], []], "negative": [[-3]], "not_list": {"a": 1}, "flat": [1, 2], "float": [[1.5]], "empty": [],
                 "long": [list(range(65))], "many": [[1]] * 1025, "ids": [[1] * 64] * 65}
    for name, content in bad_files.items():
        (tmp_path / f"{name}.json").write_text(json.dumps(content))
    (tmp_path / "broken.json").write_text("[[1, 2]")
    for bad in (["-length_penalty", "inf"], ["-length_penalty", "nan"], ["-q_length_penalty", "-inf"], ["-bad_words_ids", str(tmp_path / "nope")],
                ["-bad_words_ids", str(tmp_path / "broken.json")]) + tuple(["-q_bad_words_ids", str(tmp_path / f"{n}.json")] for n in bad_files):
        with pytest.raises(SystemExit):
            options.read_command_line(base + bad)


# ---- GPU: tiny fp32 against the oracles -------------------------------------------------------------------------------
_ORACLE = {}
_SEED = 0x5EED
_WARP = dict(temperature=0.7, top_k=7, top_p=0.0)
MODES = {"beam3": dict(num_beams=3), "beam5": dict(num_beams=5), "nbest3": dict(num_beams=3, num_return_sequences=3),
         "groups": dict(num_beams=6, num_beam_groups=3, diversity_penalty=0.5),
         "beam_sample": dict(num_beams=3, do_sample=True, num_return_sequences=2, seed=_SEED, **_WARP)}
PROCS = dict(repetition_penalty=1.3, no_repeat_ngram_size=3, min_length=9)


def _lists(prefix):
    """Bad-word lists for the tiny repetitive model (ids 300..302 and [SEP] are attractive): one-id bans, phrases, a phrase that reaches
    into the decoder prefix, and a lone [SEP] (dropped)."""
    lists = {"single": [[300], [102]], "multi": [[301, 302], [300, 301, 300], [302, 300]],
             "mixed": [[302], [300, 301], [301, 300, 300], [102], [300, 102]]}
    if prefix is not None:
        lists["into_prefix"] = [[int(prefix[0, -1]), 300], [int(prefix[1, -2]), int(prefix[1, -1]), 301], [301]]
    return lists


def _case(case):
    """(list name, processors or None, with prefix)"""
    words, _, rest = case.partition("+")
    return words, (dict(PROCS) if "procs" in rest else None), ("prefix" in rest)


CASES = ["single", "multi", "mixed", "mixed+procs", "into_prefix+prefix", "mixed+procs+prefix"]


@pytest.fixture(scope="module")
def engines(tiny_cfgs, tiny_sd):
    from gst_visdial_b200 import _lib
    from test_logits_processors import _engine
    enc_cfg, dec_cfg = tiny_cfgs
    sd = _with_bias(tiny_sd, {R.EOS: 4.0, 300: 6.0, 301: 6.0, 302: 5.5})
    b = _with_question(history_batch(enc_cfg, 0, 3), A4["tiny"])
    es = {"separate_calls": _engine(enc_cfg, dec_cfg, sd, "fp32", b),
          "no_cuda_graph": _engine(enc_cfg, dec_cfg, sd, "fp32", b, flags=_lib.GSTVD_FLAG_NO_CUDA_GRAPH)}
    es["whole_round"] = es["separate_calls"]
    yield es, b, sd
    for e in set(es.values()):
        e.close()


def _beam_oracle(sd, enc_cfg, dec_cfg, b, mode, n, words_name, words, procs, prefix):
    key = (mode, n, words_name, procs is not None, prefix is not None)
    if key not in _ORACLE:
        m = MODES[mode]
        with torch.no_grad():
            if mode == "beam_sample":
                _ORACLE[key] = DA.beam_sample(sd, enc_cfg, dec_cfg, b, m["num_beams"], m["num_return_sequences"], seed=_SEED, ngram_blocking_size=n,
                                              prefix=prefix, processors=procs, bad_words_ids=words, **_WARP)
            else:
                st = DA.group_beam_state(sd, enc_cfg, dec_cfg, b, m["num_beams"], m.get("num_beam_groups", 1), m.get("diversity_penalty", 0.0),
                                         ngram_blocking_size=n, prefix=prefix, processors=procs, bad_words_ids=words)
                _ORACLE[key] = finalize_nbest(st, m.get("num_return_sequences", 1))
    return _ORACLE[key]


def _check_no_bad_word(ids, prefix, words, per_image=1):
    for r, row in enumerate(ids.tolist()):
        d = LP.decoder_ids(prefix[r // per_image].tolist()) if prefix is not None else [R.CLS]
        out = row[:row.index(R.EOS)] if R.EOS in row else row
        assert not DA.completes_bad_word(d, out, words), (r, row)


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["separate_calls", "whole_round", "no_cuda_graph"])
@pytest.mark.parametrize("n", [0, 4])
@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("mode", sorted(MODES))
def test_tiny_fp32_beams_match_oracle(tiny_cfgs, engines, mode, case, n, path):
    from test_logits_processors import _run
    enc_cfg, dec_cfg = tiny_cfgs
    es, b, sd = engines
    words_name, procs, with_prefix = _case(case)
    pre = _prefixes(3, 5, enc_cfg.vocab_size) if with_prefix else None
    words = _lists(pre)[words_name]
    ref, ref_sc = _beam_oracle(sd, enc_cfg, dec_cfg, b, mode, n, words_name, words, procs, pre)
    _check_no_bad_word(ref, pre, words, MODES[mode].get("num_return_sequences", 1))
    ids, sc = _run(es[path], b, path, ngram_blocking_size=n, prefix=pre, bad_words_ids=words, **MODES[mode], **(procs or {}))
    assert torch.equal(ids.cpu(), ref), f"{ids.cpu().tolist()} vs {ref.tolist()}"
    tol = dict(rtol=2e-6, atol=1e-4) if mode == "beam_sample" else dict(rtol=0, atol=1e-5)
    assert torch.allclose(sc.cpu().double(), ref_sc.double(), **tol), (sc, ref_sc)


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["separate_calls", "whole_round", "no_cuda_graph"])
@pytest.mark.parametrize("n", [0, 4])
@pytest.mark.parametrize("case", CASES)
def test_tiny_fp32_greedy_matches_restatement(tiny_cfgs, engines, case, n, path):
    from test_logits_processors import _run
    enc_cfg, dec_cfg = tiny_cfgs
    es, b, sd = engines
    words_name, procs, with_prefix = _case(case)
    pre = _prefixes(3, 5, enc_cfg.vocab_size) if with_prefix else None
    words = _lists(pre)[words_name]
    key = ("greedy", n, case)
    if key not in _ORACLE:
        bb = dict(b, dec_input_ids=pre if pre is not None else b["dec_input_ids"])
        with torch.no_grad():
            _ORACLE[key] = DA.generate_greedy_or_sample(sd, enc_cfg, dec_cfg, bb, 1.0, 1, 0.0, n, processors=procs, bad_words_ids=words)
    ref = _ORACLE[key]
    _check_no_bad_word(ref, pre, words)
    ids, _ = _run(es[path], b, path, top_k=1, ngram_blocking_size=n, prefix=pre, bad_words_ids=words, **(procs or {}))
    assert torch.equal(ids.cpu(), ref), (ids.cpu().tolist(), ref.tolist())


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["separate_calls", "whole_round", "no_cuda_graph"])
@pytest.mark.parametrize("top_k", [7, 0])
@pytest.mark.parametrize("case", ["mixed", "mixed+procs", "into_prefix+prefix"])
def test_tiny_fp32_sampling_never_completes_a_listed_sequence(tiny_cfgs, engines, case, top_k, path):
    """top-k 7 and top_k = 0 samples: no listed sequence completed, every token inside the processed (bad words included) support."""
    from test_logits_processors import _run
    enc_cfg, dec_cfg = tiny_cfgs
    es, b, sd = engines
    words_name, procs, with_prefix = _case(case)
    pre = _prefixes(3, 5, enc_cfg.vocab_size) if with_prefix else None
    words = _lists(pre)[words_name]
    p = dict(dict(repetition_penalty=1.0, no_repeat_ngram_size=0, min_length=0), **(procs or {}))
    for seed in (_SEED, _SEED + 1):
        ids, _ = _run(es[path], b, path, temperature=0.7, top_k=top_k, prefix=pre, seed=seed, num_return_sequences=2, bad_words_ids=words, **p)
        ids = ids.cpu()
        _check_no_bad_word(ids, pre, words, 2)
        bb = {k: v.repeat_interleave(2, 0) if torch.is_tensor(v) else v for k, v in b.items()}
        start = pre.repeat_interleave(2, 0) if pre is not None else bb["dec_input_ids"]
        dec = torch.cat((start, ids), 1)
        with torch.no_grad():
            seq_t, seq_v = R.encoder(sd, enc_cfg, bb["enc_input_ids"], bb["enc_image_feat"], bb["enc_image_loc"], bb["enc_segments"],
                                     bb["enc_att_mask"], bb["enc_image_mask"])
            enc_h, enc_m = R.vlfusion(sd, seq_t, seq_v, bb["enc_att_mask"], bb["enc_image_mask"])
            _, logits = R.decoder_forward(sd, dec_cfg, dec.clone(), None, enc_h, enc_m)
        P = start.shape[1]
        for t in range(ids.shape[1]):
            d_rows = [LP.decoder_ids(r) for r in dec[:, :P + t].tolist()]
            step = DA.apply(logits[:, P - 1 + t, :] / 0.7, d_rows, p, words)
            step = R.top_k_top_p_filter(step, top_k, 0.0)
            for r in range(ids.shape[0]):
                if R.EOS not in ids[r, :t].tolist():
                    assert step[r, ids[r, t]] > -float("inf"), (r, t, int(ids[r, t]))


@pytest.mark.gpu
@pytest.mark.parametrize("top_k", [1, 7, 0])
def test_op_sample_honours_the_list(tiny_cfgs, tiny_sd, top_k):
    from gst_visdial_b200.engine import Engine
    enc_cfg, dec_cfg = tiny_cfgs
    e = Engine(enc_cfg, dec_cfg, dtype="fp32", max_batch=8, max_beams=5)
    try:
        e.load_state_dict(tiny_sd)
        rows, V, step = 8, enc_cfg.vocab_size, 6
        g = torch.Generator().manual_seed(12)
        logits = torch.randn(rows, V, generator=g)
        prefix = torch.randint(300, 304, (rows, step + 1), generator=g)
        prefix[:, 0] = R.CLS
        logits[:, 300:306] += 9.0                                    # the listed ids would win without the list
        words = [[300], [301, 302], [int(prefix[0, -1]), 303], list(map(int, prefix[1])) + [304], [102]]
        proc = DA.apply_bad_words(logits, [LP.decoder_ids(r) for r in prefix.tolist()], words)
        assert (proc[1, 304] == -float("inf")) and (proc[0, 303] == -float("inf"))
        for seed in range(4 if top_k != 1 else 1):
            out = e.op_sample(logits.cuda(), step, temperature=1.0, top_k=top_k, seed=seed, prefix=prefix.cuda(), bad_words_ids=words).cpu().long()
            if top_k == 1:
                assert torch.equal(out, proc.argmax(-1)), (out, proc.argmax(-1))
            else:
                assert bool((R.top_k_top_p_filter(proc, top_k, 0.0).gather(1, out[:, None]) > -float("inf")).all()), out
    finally:
        e.close()


@pytest.mark.gpu
def test_graph_cache_replays_the_current_list(tiny_cfgs, engines):
    """Lists of the same shape with different ids share a graph and each call follows its own list; a new shape captures anew."""
    from test_logits_processors import _run
    enc_cfg, dec_cfg = tiny_cfgs
    es, b, sd = engines
    e = es["separate_calls"]
    lists = {"a": [[300], [301, 302]], "b": [[301], [300, 302]], "c": [[302], [301, 300]], "d": [[300], [302], [301, 300]]}
    for name in ("a", "b", "a", "c", "d", "b"):
        words = lists[name]
        for mode in ("beam3", "greedy"):
            key = ("cache", mode, name)
            if key not in _ORACLE:
                with torch.no_grad():
                    if mode == "greedy":
                        _ORACLE[key] = DA.generate_greedy_or_sample(sd, enc_cfg, dec_cfg, b, 1.0, 1, 0.0, 0, bad_words_ids=words)
                    else:
                        _ORACLE[key] = DA.group_beam_state(sd, enc_cfg, dec_cfg, b, 3, bad_words_ids=words).finalize()[0]
            kw = dict(top_k=1) if mode == "greedy" else MODES["beam3"]
            ids, _ = _run(e, b, "separate_calls", bad_words_ids=words, **kw)
            assert torch.equal(ids.cpu(), _ORACLE[key]), (name, mode)
            ids, _ = _run(e, b, "whole_round", bad_words_ids=words, **kw)
            assert torch.equal(ids.cpu(), _ORACLE[key]), (name, mode, "round")


@pytest.mark.gpu
def test_rejections(tiny_cfgs, tiny_sd):
    from gst_visdial_b200 import _lib
    from gst_visdial_b200._lib import GstvdError
    from test_logits_processors import _engine
    enc_cfg, dec_cfg = tiny_cfgs
    b = history_batch(enc_cfg, 0, 2)
    e = _engine(enc_cfg, dec_cfg, tiny_sd, "fp32", b)
    V = enc_cfg.vocab_size
    bad = [[[]], [[V]], [[-5]], [list(range(1, 66))], [[1]] * 1025, [[1] * 64] * 65]
    try:
        for mode in (dict(), dict(num_beams=3), dict(num_beams=3, do_sample=True, top_k=7)):
            for words in bad:
                with pytest.raises(GstvdError) as ei:
                    e.generate(2, bad_words_ids=words, **mode)
                assert ei.value.status == -1, words
        for words in bad[:3]:
            with pytest.raises(GstvdError):
                e.op_sample(torch.zeros(2, V, device="cuda"), 0, prefix=torch.full((2, 1), 101, device="cuda"), bad_words_ids=words)
        # the caps themselves are accepted
        e.generate(2, num_beams=3, bad_words_ids=[[1] * 64] * 64)
        e.generate(2, bad_words_ids=[[w % V] for w in range(1024)])
        out = torch.empty(2, 18, dtype=torch.int64, device="cuda:0")
        gp = e._gen_params(num_beams=3)
        for ids, n in (((ctypes.c_int32 * 2)(5, 7), 2), (None, 3)):      # not closed by -1; a length without an address
            gp.bad_words_ids = ctypes.addressof(ids) if ids is not None else 0
            gp.bad_words_len = n
            assert e.lib.gstvd_generate(e.ctx, 2, ctypes.byref(gp), None, 1, None, None, 0, ctypes.c_void_p(out.data_ptr()), None, e._stream()) == -1
        gp.bad_words_len = -1
        assert e.lib.gstvd_generate(e.ctx, 2, ctypes.byref(gp), None, 1, None, None, 0, ctypes.c_void_p(out.data_ptr()), None, e._stream()) == -1
        assert _lib.GSTVD_ABI_VERSION == 7
    finally:
        e.close()


# ---- GPU: full config, bf16 ------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_full_bf16_off_path_and_properties(full_cfgs, full_sd):
    """Everything off: the same bits whether the defaults are passed or not, and 1857 kernels per beam-5 call; with the features on
    the launch count is unchanged and no output completes a listed sequence."""
    from test_logits_processors import _engine, _run
    enc_cfg, dec_cfg = full_cfgs
    b = history_batch(enc_cfg, 0, 4)
    e = _engine(enc_cfg, dec_cfg, full_sd, "bf16", b)
    try:
        with torch.no_grad():
            greedy = LP.generate_greedy_or_sample(full_sd, enc_cfg, dec_cfg, b, 1.0, 1, 0.0, 0, max_new=6)
        words = [[int(w)] for w in greedy[:, 0].tolist()] + [[int(greedy[r, 0]), int(greedy[r, 1])] for r in range(4)] + [[102]]
        for kw in (dict(num_beams=5), dict(temperature=0.7, top_k=7, seed=3, ngram_blocking_size=4), dict(temperature=0.7, top_k=0, seed=3),
                   dict(num_beams=4, do_sample=True, temperature=0.7, top_k=7, seed=3), dict(num_beams=6, num_beam_groups=3, diversity_penalty=0.5)):
            ids0, sc0 = _run(e, b, "separate_calls", **kw)
            ids1, sc1 = _run(e, b, "separate_calls", bad_words_ids=[], length_penalty=1.0, early_stopping=False, **kw)
            assert torch.equal(ids0, ids1) and (kw.get("num_beams", 1) == 1 or torch.equal(sc0, sc1)), kw   # sampling writes no scores
            for path in ("separate_calls", "whole_round"):
                ids, _ = _run(e, b, path, bad_words_ids=words, repetition_penalty=1.2, **kw)
                _check_no_bad_word(ids.cpu(), None, words, ids.shape[0] // 4)
        for n, want in ((0, 1857), (4, 1872)):
            for kw in (dict(), dict(bad_words_ids=words, length_penalty=1.5, early_stopping=True)):
                before = e.launch_count
                e.generate(4, num_beams=5, ngram_blocking_size=n, hist_ids=b["enc_input_ids"], hist_segments=b["enc_segments"], **kw)
                torch.cuda.synchronize()
                assert e.launch_count - before == want, (n, kw, e.launch_count - before)
    finally:
        e.close()


@pytest.mark.gpu
def test_generate_cli_with_the_new_flags(tmp_path):
    import subprocess
    import sys
    words = [[2054], [2064, 2017]]
    f = tmp_path / "bw.json"
    f.write_text(json.dumps(words))
    cmd = [sys.executable, os.path.join(ROOT, "generate.py"), "-synthetic", "8", "-batch_size", "8", "-num_rounds", "2", "-num_beams", "3",
           "-length_penalty", "1.5", "-early_stopping", "-bad_words_ids", str(f), "-q_bad_words_ids", str(f), "-q_length_penalty", "0.8",
           "-save_path", str(tmp_path), "-save_name", "o.json"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout + r.stderr
    out = json.load(open(tmp_path / "o.json"))
    assert len(out) >= 1 and all(len(d["dialog"]) == 2 for d in out)
    ids = lambda u: [int(x) for x in u.split()] if isinstance(u, str) else [int(x) for x in u]     # noqa: E731
    for d in out:
        for turn in d["dialog"]:
            for u in (turn["answer"], turn["question"]):
                assert not DA.completes_bad_word([R.CLS], [w for w in ids(u) if w != R.EOS], words), turn
