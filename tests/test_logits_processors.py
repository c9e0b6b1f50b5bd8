"""HF logits processors in every decode mode: repetition_penalty, no_repeat_ngram_size and min_length (include/gstvd.h gstvd_generate,
CPU oracle oracle/processors.py, pinned on HF's own classes by oracle/gen_golden_processors.py)."""
import ctypes
import os

import numpy as np
import pytest
import torch

from helpers import ROOT, R, history_batch
from oracle import beam_groups as BG
from oracle import beam_ngram as BN
from oracle import beam_sample as BS
from oracle import processors as LP
from test_decoder_prefix import _prefixes

GOLDEN = os.path.join(ROOT, "tests", "golden", "logits_processors.npz")
OFF = dict(repetition_penalty=1.0, no_repeat_ngram_size=0, min_length=0)
PROCS = {"rep": dict(repetition_penalty=1.3), "ngram": dict(no_repeat_ngram_size=2), "minlen": dict(min_length=9),
         "all": dict(repetition_penalty=1.3, no_repeat_ngram_size=3, min_length=9)}


def _full(p):
    return dict(OFF, **p)


# ---- CPU: the restatement ------------------------------------------------------------------------------------------
def _golden_cases():
    g = np.load(GOLDEN)
    names = sorted({k.rsplit("_", 1)[0] for k in g.files})
    for n in names:
        p, ng, m = g[f"{n}_params"]
        yield n, torch.from_numpy(g[f"{n}_scores"]), torch.from_numpy(g[f"{n}_ids"]), float(p), int(ng), int(m), torch.from_numpy(g[f"{n}_out"])


def test_restatement_equals_goldens():
    cases = list(_golden_cases())
    assert len(cases) >= 16
    assert {c[4] for c in cases} >= {0, 1, 2, 3} and any(c[4] > c[2].shape[1] for c in cases)      # n = 1 and n longer than d
    for name, s, ids, p, n, m, out in cases:
        ours = LP.apply(s, ids.tolist(), repetition_penalty=p, no_repeat_ngram_size=n, min_length=m)
        assert torch.equal(ours, out), name


def test_restatement_equals_hf():
    pytest.importorskip("transformers")
    from oracle.gen_golden_processors import cases, hf_apply
    for name, s, ids, p, n, m in cases():
        assert torch.equal(LP.apply(s, ids.tolist(), repetition_penalty=p, no_repeat_ngram_size=n, min_length=m), hf_apply(s, ids, p, n, m)), name


def test_repeated_id_is_penalised_once():
    s = torch.tensor([[2.0, -2.0, 3.0, -float("inf"), 1.0]])
    out = LP.apply(s, [[0, 0, 0, 1, 1, 3]], repetition_penalty=2.0)
    assert out.tolist() == [[1.0, -4.0, 3.0, -float("inf"), 1.0]]


def test_ngram_rule_examples():
    assert LP.no_repeat_ngram_banned([101, 5, 6, 5], 2) == [6]
    assert sorted(LP.no_repeat_ngram_banned([101, 5, 6], 1)) == [5, 6, 101]
    assert LP.no_repeat_ngram_banned([5, 6, 5], 5) == []
    assert LP.no_repeat_ngram_banned([7, 8, 7, 8, 7], 3) == [8]


def _random_steps(rows, V, T, seed):
    g = torch.Generator().manual_seed(seed)
    return [torch.randn(rows, V, generator=g) * 3.0 for _ in range(T)]


@pytest.mark.parametrize("cls", ["blocked", "groups", "sample"])
def test_hooked_oracles_off_are_unchanged(cls):
    B, K, V, T = 2, 4, 300, 10
    steps = _random_steps(B * K * (2 if cls == "sample" else 1), V, T, 3)
    for s in steps:
        s[:, R.EOS] += 2.0
    base, processed = {"blocked": (lambda: BN.BlockedBeamState(B, K, V, T), lambda: LP.ProcessedGroupBeamState(B, K, V, T, processors=OFF)),
                       "groups": (lambda: BG.GroupBeamState(B, K, V, T, num_beam_groups=2, diversity_penalty=0.5),
                                  lambda: LP.ProcessedGroupBeamState(B, K, V, T, num_beam_groups=2, diversity_penalty=0.5, processors=OFF)),
                       "sample": (lambda: BS.BeamSampleState(B, K, V, T, N=2, seed=7),
                                  lambda: LP.ProcessedBeamSampleState(B, K, V, T, N=2, seed=7, processors=OFF))}[cls]
    a, b = base(), processed()
    for lg in steps:
        ra, rb = a.step(lg), b.step(lg)
        assert all(torch.equal(x, y) for x, y in zip(ra, rb))
    fa, fb = a.finalize(), b.finalize()
    assert all(torch.equal(x, y) for x, y in zip(fa, fb))


def test_restatement_off_is_unchanged(tiny_cfgs, tiny_sd):
    enc_cfg, dec_cfg = tiny_cfgs
    b = history_batch(enc_cfg, 0, 2)
    with torch.no_grad():
        a = R.generate_greedy_or_sample(tiny_sd, enc_cfg, dec_cfg, b, 1.0, 1, 0.0, 4, max_new=6)
        c = LP.generate_greedy_or_sample(tiny_sd, enc_cfg, dec_cfg, b, 1.0, 1, 0.0, 4, max_new=6, processors=dict(OFF))
    assert torch.equal(a, c)


def _until_sep(row):
    out = []
    for w in row:
        if int(w) == R.EOS:
            break
        out.append(int(w))
    return out


def _first_sep(row):
    row = [int(w) for w in row]
    return row.index(R.EOS) if R.EOS in row else len(row)


def _check_properties(seqs, prefix, p, B, per_image=1):
    """n-gram / min-length properties of output rows given the rows' decoder prefix ([B, P] or None)."""
    for r, row in enumerate(seqs.tolist()):
        d = LP.decoder_ids(prefix[r // per_image].tolist()) if prefix is not None else [R.CLS]
        P = len(d)
        if p.get("no_repeat_ngram_size", 0):
            assert not LP.has_repeated_ngram(d + _until_sep(row), p["no_repeat_ngram_size"]), (r, row)
        if p.get("min_length", 0):
            assert _first_sep(row) >= p["min_length"] - P, (r, row)


@pytest.fixture(scope="module")
def repetitive_sd(tiny_sd):
    """Tiny weights whose LM head favours a few ids and [SEP]: without the processors the output repeats itself and ends early."""
    from test_decoder_prefix import _with_bias
    return _with_bias(tiny_sd, {R.EOS: 4.0, 300: 6.0, 301: 6.0, 302: 5.5})


@pytest.mark.parametrize("case", sorted(PROCS))
def test_oracle_properties_on_tiny_model(tiny_cfgs, repetitive_sd, case):
    enc_cfg, dec_cfg = tiny_cfgs
    p = _full(PROCS[case])
    b = history_batch(enc_cfg, 0, 2)
    with torch.no_grad():
        g = LP.generate_greedy_or_sample(repetitive_sd, enc_cfg, dec_cfg, b, 1.0, 1, 0.0, 0, max_new=12, processors=p)
        st = LP.group_beam_state(repetitive_sd, enc_cfg, dec_cfg, b, 3, max_new=12, processors=p)
        beams, _ = st.finalize()
    _check_properties(g, None, p, 2)
    _check_properties(beams, None, p, 2)
    if case == "all":
        with torch.no_grad():
            g0 = R.generate_greedy_or_sample(repetitive_sd, enc_cfg, dec_cfg, b, 1.0, 1, 0.0, 0, max_new=12)
        assert any(LP.has_repeated_ngram([R.CLS] + _until_sep(r), 3) or _first_sep(r) < 8 for r in g0.tolist())   # the case is not vacuous


def test_cli_flags(tmp_path):
    from gst_visdial_b200 import options
    base = ["-save_path", str(tmp_path)]
    p = options.read_command_line(base)
    assert (p["repetition_penalty"], p["no_repeat_ngram_size"], p["min_length"]) == (1.0, 0, 0)
    assert (p["q_repetition_penalty"], p["q_no_repeat_ngram_size"], p["q_min_length"]) == (1.0, 0, 0)
    p = options.read_command_line(base + ["-repetition_penalty", "1.2", "-no_repeat_ngram_size", "3", "-min_length", "4",
                                          "-q_repetition_penalty", "0.9", "-q_no_repeat_ngram_size", "2", "-q_min_length", "6"])
    assert (p["repetition_penalty"], p["no_repeat_ngram_size"], p["min_length"]) == (1.2, 3, 4)
    assert (p["q_repetition_penalty"], p["q_no_repeat_ngram_size"], p["q_min_length"]) == (0.9, 2, 6)
    for bad in (["-repetition_penalty", "0"], ["-repetition_penalty", "-1"], ["-repetition_penalty", "inf"], ["-repetition_penalty", "nan"],
                ["-no_repeat_ngram_size", "-1"], ["-min_length", "-2"], ["-q_repetition_penalty", "0"], ["-q_no_repeat_ngram_size", "-1"],
                ["-q_min_length", "-1"]):
        with pytest.raises(SystemExit):
            options.read_command_line(base + bad)


# ---- GPU: tiny fp32 against the oracles -----------------------------------------------------------------------------
_ORACLE = {}
_SEED = 0x5EED
_WARP = dict(temperature=0.7, top_k=7, top_p=0.0)
MODES = {"beam3": dict(num_beams=3), "beam5": dict(num_beams=5), "groups": dict(num_beams=6, num_beam_groups=3, diversity_penalty=0.5),
         "beam_sample": dict(num_beams=3, do_sample=True, num_return_sequences=2, seed=_SEED, **_WARP)}
CASES = ["rep", "ngram", "minlen", "all", "all_prefix"]


def _case(case):
    return _full(PROCS[case.replace("_prefix", "")]), (case.endswith("_prefix"))


def _tiny_batch(enc_cfg):
    from test_decoder_prefix import A4, _with_question
    return _with_question(history_batch(enc_cfg, 0, 3), A4["tiny"])


def _beam_oracle(sd, enc_cfg, dec_cfg, b, mode, n, p, prefix):
    key = (mode, n, tuple(sorted(p.items())), prefix is not None)
    if key not in _ORACLE:
        m = MODES[mode]
        with torch.no_grad():
            if mode == "beam_sample":
                _ORACLE[key] = LP.beam_sample(sd, enc_cfg, dec_cfg, b, m["num_beams"], m["num_return_sequences"], seed=_SEED,
                                              ngram_blocking_size=n, prefix=prefix, processors=p, **_WARP)
            else:
                st = LP.group_beam_state(sd, enc_cfg, dec_cfg, b, m["num_beams"], m.get("num_beam_groups", 1), m.get("diversity_penalty", 0.0),
                                         ngram_blocking_size=n, prefix=prefix, processors=p)
                _ORACLE[key] = st.finalize()
    return _ORACLE[key]


def _engine(enc_cfg, dec_cfg, sd, dtype, b, flags=0):
    from gst_visdial_b200.engine import Engine
    B = b["enc_input_ids"].shape[0]
    e = Engine(enc_cfg, dec_cfg, dtype=dtype, max_batch=B, max_beams=8, flags=flags)
    e.load_state_dict(sd)
    o = e.encode(b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"], b["enc_image_mask"])
    e.prefill_cross(B, o["Le"])
    return e


def _run(e, b, path, **kw):
    """(ids, scores) of one decode request through the path: separate calls / the whole-round graph / eager (engine flag)."""
    B = b["enc_input_ids"].shape[0]
    if path == "whole_round":
        return e.round(b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"], b["enc_image_mask"],
                       want_scores=True, **kw)
    return e.generate(B, want_scores=True, hist_ids=b["enc_input_ids"], hist_segments=b["enc_segments"], **kw)


@pytest.fixture(scope="module")
def engines(tiny_cfgs, repetitive_sd):
    from gst_visdial_b200 import _lib
    enc_cfg, dec_cfg = tiny_cfgs
    b = _tiny_batch(enc_cfg)
    es = {"separate_calls": _engine(enc_cfg, dec_cfg, repetitive_sd, "fp32", b), "no_cuda_graph":
          _engine(enc_cfg, dec_cfg, repetitive_sd, "fp32", b, flags=_lib.GSTVD_FLAG_NO_CUDA_GRAPH)}
    es["whole_round"] = es["separate_calls"]
    yield es, b
    for e in set(es.values()):
        e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["separate_calls", "whole_round", "no_cuda_graph"])
@pytest.mark.parametrize("n", [0, 4])
@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("mode", sorted(MODES))
def test_tiny_fp32_beams_match_oracle(tiny_cfgs, repetitive_sd, engines, mode, case, n, path):
    enc_cfg, dec_cfg = tiny_cfgs
    es, b = engines
    p, with_prefix = _case(case)
    pre = _prefixes(3, 5, enc_cfg.vocab_size) if with_prefix else None
    ref, ref_sc = _beam_oracle(repetitive_sd, enc_cfg, dec_cfg, b, mode, n, p, pre)
    _check_properties(ref, pre, p, 3, MODES[mode].get("num_return_sequences", 1))
    ids, sc = _run(es[path], b, path, ngram_blocking_size=n, prefix=pre, **MODES[mode], **p)
    assert torch.equal(ids.cpu(), ref), f"{ids.cpu().tolist()} vs {ref.tolist()}"
    # beam sampling divides every step's scores by the temperature again, so a last-bit difference of an early logZ (the kernel's
    # table-driven fp64 exp) grows with the length: a relative bound there, as in test_beam_sample
    tol = dict(rtol=2e-6, atol=1e-4) if mode == "beam_sample" else dict(rtol=0, atol=1e-5)
    assert torch.allclose(sc.cpu().double(), ref_sc.double(), **tol), (sc, ref_sc)


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["separate_calls", "whole_round", "no_cuda_graph"])
@pytest.mark.parametrize("n", [0, 4])
@pytest.mark.parametrize("case", CASES)
def test_tiny_fp32_greedy_matches_restatement(tiny_cfgs, repetitive_sd, engines, case, n, path):
    enc_cfg, dec_cfg = tiny_cfgs
    es, b = engines
    p, with_prefix = _case(case)
    pre = _prefixes(3, 5, enc_cfg.vocab_size) if with_prefix else None
    key = ("greedy", n, tuple(sorted(p.items())), with_prefix)
    if key not in _ORACLE:
        bb = dict(b, dec_input_ids=pre if pre is not None else b["dec_input_ids"])
        with torch.no_grad():
            _ORACLE[key] = LP.generate_greedy_or_sample(repetitive_sd, enc_cfg, dec_cfg, bb, 1.0, 1, 0.0, n, processors=p)
    ref = _ORACLE[key]
    ids, _ = _run(es[path], b, path, top_k=1, ngram_blocking_size=n, prefix=pre, **p)
    ids = ids.cpu()
    for r in range(ids.shape[0]):               # the engine writes PAD after the first [SEP]; so does the restatement
        assert ids[r].tolist() == ref[r].tolist(), (r, ids[r].tolist(), ref[r].tolist())


def _support_check(sd, enc_cfg, dec_cfg, b, ids, pre, n, p, temperature, top_k):
    """Teacher-forced: every sampled token up to the first [SEP] lies in the support of the processed, top-k-filtered row."""
    B, T = ids.shape
    start = pre if pre is not None else b["dec_input_ids"]
    dec = torch.cat((start, ids), 1)
    seq_t, seq_v = R.encoder(sd, enc_cfg, b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"],
                             b["enc_image_mask"])
    enc_h, enc_m = R.vlfusion(sd, seq_t, seq_v, b["enc_att_mask"], b["enc_image_mask"])
    _, logits = R.decoder_forward(sd, dec_cfg, dec.clone(), None, enc_h, enc_m)
    hist = (b["enc_input_ids"] * (b["enc_segments"] == 0).long()).tolist()
    P = start.shape[1]
    checked = 0
    for t in range(T):
        step = logits[:, P - 1 + t, :] / temperature
        step = LP.apply(step, [LP.decoder_ids(r) for r in dec[:, :P + t].tolist()], **p)
        for r in range(B):
            for w in R.ngram_banned_tokens(hist[r], dec[r, :P + t].tolist(), n) if n else []:
                step[r, w] = -float("inf")
        step = R.top_k_top_p_filter(step, top_k, 0.0)
        for r in range(B):
            if R.EOS in ids[r, :t].tolist():
                continue
            assert step[r, ids[r, t]] > -float("inf"), (r, t, int(ids[r, t]))
            checked += 1
    assert checked >= B


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["separate_calls", "whole_round", "no_cuda_graph"])
@pytest.mark.parametrize("top_k", [7, 0])
@pytest.mark.parametrize("case", ["rep", "ngram", "minlen", "all", "all_prefix", "all_hist"])
def test_tiny_fp32_sampling_stays_in_processed_support(tiny_cfgs, repetitive_sd, engines, case, top_k, path):
    enc_cfg, dec_cfg = tiny_cfgs
    es, b = engines
    n = 4 if case == "all_hist" else 0
    p, with_prefix = _case(case.replace("_hist", ""))
    pre = _prefixes(3, 5, enc_cfg.vocab_size) if with_prefix else None
    ids, _ = _run(es[path], b, path, temperature=0.7, top_k=top_k, ngram_blocking_size=n, prefix=pre, seed=_SEED, num_return_sequences=2, **p)
    ids = ids.cpu()
    _check_properties(ids, pre, p, 3, 2)
    with torch.no_grad():
        bb = {k: v.repeat_interleave(2, 0) if torch.is_tensor(v) else v for k, v in b.items()}
        _support_check(repetitive_sd, enc_cfg, dec_cfg, bb, ids, pre.repeat_interleave(2, 0) if pre is not None else None, n, p, 0.7, top_k)


@pytest.mark.gpu
@pytest.mark.parametrize("top_k", [1, 7, 0])
def test_op_sample_matches_hf_processed_logits(tiny_cfgs, tiny_sd, top_k):
    enc_cfg, dec_cfg = tiny_cfgs
    from gst_visdial_b200.engine import Engine
    e = Engine(enc_cfg, dec_cfg, dtype="fp32", max_batch=8, max_beams=5)
    try:
        e.load_state_dict(tiny_sd)
        rows, V, step = 8, enc_cfg.vocab_size, 9
        g = torch.Generator().manual_seed(11)
        logits = torch.randn(rows, V, generator=g) * 2.0
        prefix = torch.randint(300, 306, (rows, step + 1), generator=g)           # a small alphabet: ids and 2-grams repeat
        prefix[:, 0] = R.CLS
        prefix[0, 3] = R.EOS
        logits[:, 300:306] += 6.0                                                   # the history ids would win without the penalty
        logits[:, R.EOS] += 8.0
        p = dict(repetition_penalty=1.7, no_repeat_ngram_size=2, min_length=14)
        proc = LP.apply(logits, [LP.decoder_ids(r) for r in prefix.tolist()], **p)
        for seed in range(4 if top_k != 1 else 1):
            out = e.op_sample(logits.cuda(), step, temperature=1.0, top_k=top_k, seed=seed, prefix=prefix.cuda(), **p).cpu().long()
            if top_k == 1:
                assert torch.equal(out, proc.argmax(-1)), (out, proc.argmax(-1))
            else:
                filt = R.top_k_top_p_filter(proc, top_k, 0.0)
                assert bool((filt.gather(1, out[:, None]) > -float("inf")).all()), out
            assert not bool((out == R.EOS).any())
        with pytest.raises(Exception):
            e.op_sample(logits.cuda(), step, top_k=top_k, prefix=prefix[:, :3].cuda(), **p)        # prefix must hold step + 1 ids
    finally:
        e.close()


@pytest.mark.gpu
def test_graph_cache_keys_the_processors(tiny_cfgs, repetitive_sd, engines):
    enc_cfg, dec_cfg = tiny_cfgs
    es, b = engines
    e = es["separate_calls"]
    for case in ("rep", "ngram", "all", "rep", "minlen"):
        p = _full(PROCS[case])
        ref, ref_sc = _beam_oracle(repetitive_sd, enc_cfg, dec_cfg, b, "beam3", 0, p, None)
        ids, sc = _run(e, b, "separate_calls", ngram_blocking_size=0, **MODES["beam3"], **p)
        assert torch.equal(ids.cpu(), ref), case
    ref, _ = _beam_oracle(repetitive_sd, enc_cfg, dec_cfg, b, "beam3", 0, dict(OFF), None)
    ids, _ = _run(e, b, "separate_calls", ngram_blocking_size=0, **MODES["beam3"])
    assert torch.equal(ids.cpu(), ref)


@pytest.mark.gpu
def test_rejections(tiny_cfgs, tiny_sd):
    from gst_visdial_b200 import _lib
    from gst_visdial_b200._lib import GstvdError
    enc_cfg, dec_cfg = tiny_cfgs
    b = history_batch(enc_cfg, 0, 2)
    e = _engine(enc_cfg, dec_cfg, tiny_sd, "fp32", b)
    rnd = (b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"], b["enc_image_mask"])
    bad = [dict(repetition_penalty=0.0), dict(repetition_penalty=-1.0), dict(repetition_penalty=float("inf")),
           dict(repetition_penalty=float("nan")), dict(no_repeat_ngram_size=-1), dict(min_length=-1)]
    try:
        for mode in (dict(), dict(num_beams=3), dict(num_beams=3, do_sample=True, top_k=7)):
            for kw in bad:
                with pytest.raises(GstvdError) as ei:
                    e.generate(2, **mode, **kw)
                assert ei.value.status == -1, kw
                with pytest.raises(GstvdError) as ei:
                    e.round(*rnd, **mode, **kw)
                assert ei.value.status == -1, kw
        # a zero-filled params struct (every other field valid) is refused
        gp = _lib.GstvdGenParams()
        gp.mode, gp.num_beams, gp.max_new_tokens, gp.top_k, gp.temperature = _lib.GSTVD_SELECT_SAMPLE, 1, 18, 1, 1.0
        gp.num_return_sequences = gp.num_beam_groups = 1
        out = torch.empty(2, 18, dtype=torch.int64, device="cuda:0")
        assert e.lib.gstvd_generate(e.ctx, 2, ctypes.byref(gp), None, 1, None, None, 0, ctypes.c_void_p(out.data_ptr()), None, e._stream()) == -1
        gp.repetition_penalty = 1.0
        assert e.lib.gstvd_generate(e.ctx, 2, ctypes.byref(gp), None, 1, None, None, 0, ctypes.c_void_p(out.data_ptr()), None, e._stream()) == 0
    finally:
        e.close()


# ---- GPU: full config, bf16 ------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_full_bf16_processors(full_cfgs, full_sd):
    """Questioner-style (top-k 7 sampling with 4-gram question blocking, and beam-5) and teacher-style (beam-5) decoding with all three
    processors on: the properties hold; greedy ids agree with the fp32 restatement as the bf16 smoke test asks (>= 50 %)."""
    enc_cfg, dec_cfg = full_cfgs
    b = history_batch(enc_cfg, 0, 4)
    B = 4
    p = dict(repetition_penalty=1.3, no_repeat_ngram_size=3, min_length=7)
    e = _engine(enc_cfg, dec_cfg, full_sd, "bf16", b)
    try:
        for kw in (dict(temperature=0.7, top_k=7, ngram_blocking_size=4, seed=3), dict(num_beams=5, ngram_blocking_size=4), dict(num_beams=5),
                   dict(num_beams=4, do_sample=True, temperature=0.7, top_k=7, seed=3), dict(num_beams=6, num_beam_groups=3, diversity_penalty=0.5)):
            ids, _ = _run(e, b, "whole_round", **kw, **p)
            _check_properties(ids.cpu(), None, p, B)
        greedy, _ = _run(e, b, "separate_calls", top_k=1, **p)
    finally:
        e.close()
    with torch.no_grad():
        ref = LP.generate_greedy_or_sample(full_sd, enc_cfg, dec_cfg, b, 1.0, 1, 0.0, 0, processors=p)
    assert (greedy.cpu() == ref).float().mean().item() >= 0.5, (greedy, ref)


@pytest.mark.gpu
def test_full_bf16_processors_off_launch_counts(full_cfgs, full_sd):
    """Processors off: an 18-step beam-5 call launches what it did before (1857 kernels, 1872 with 4-gram blocking); on, the same."""
    enc_cfg, dec_cfg = full_cfgs
    b = history_batch(enc_cfg, 0, 4)
    e = _engine(enc_cfg, dec_cfg, full_sd, "bf16", b)
    try:
        for n, want in ((0, 1857), (4, 1872)):
            for p in (dict(), dict(OFF), dict(repetition_penalty=1.3, no_repeat_ngram_size=3, min_length=7)):
                before = e.launch_count
                e.generate(4, num_beams=5, ngram_blocking_size=n, hist_ids=b["enc_input_ids"], hist_segments=b["enc_segments"], **p)
                torch.cuda.synchronize()
                assert e.launch_count - before == want, (n, p, e.launch_count - before)
    finally:
        e.close()


@pytest.mark.gpu
def test_generate_cli_with_processors(tmp_path):
    import json
    import subprocess
    import sys
    cmd = [sys.executable, os.path.join(ROOT, "generate.py"), "-synthetic", "8", "-batch_size", "8", "-num_rounds", "2", "-num_beams", "3",
           "-no_repeat_ngram_size", "2", "-repetition_penalty", "1.2", "-min_length", "4", "-q_no_repeat_ngram_size", "3",
           "-q_min_length", "5", "-save_path", str(tmp_path), "-save_name", "o.json"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout + r.stderr
    out = json.load(open(tmp_path / "o.json"))
    assert len(out) >= 1 and all(len(d["dialog"]) == 2 for d in out)
    ids = lambda u: [int(x) for x in u.split()] if isinstance(u, str) else [int(x) for x in u]     # noqa: E731
    for d in out:
        for turn in d["dialog"]:
            assert not LP.has_repeated_ngram([R.CLS] + ids(turn["answer"]), 2), turn
            assert not LP.has_repeated_ngram([R.CLS] + ids(turn["question"]), 3), turn
