"""HF length_penalty and early_stopping in the beam modes (include/gstvd.h gstvd_generate, CPU oracle oracle/decode_args.py)."""
import copy
import math

import numpy as np
import pytest
import torch

from helpers import R, history_batch
from oracle import decode_args as DA
from oracle import processors as LP
from oracle.beam_nbest import finalize_nbest
from test_decoder_prefix import A4, _with_bias, _with_question

LAMBDAS = [0.0, 0.6, 2.0, -0.5]


# ---- CPU: the oracles -----------------------------------------------------------------------------------------------
def _random_steps(rows, V, T, seed):
    g = torch.Generator().manual_seed(seed)
    steps = [torch.randn(rows, V, generator=g) * 3.0 for _ in range(T)]
    for s in steps:
        s[:, R.EOS] += 2.0
    return steps


_STATES = {"beam": (lambda: LP.ProcessedGroupBeamState(2, 4, 300, 10, prefix=torch.tensor([[101, 7, 8], [101, 9, 102]])),
                    lambda **kw: DA.ArgsGroupBeamState(2, 4, 300, 10, prefix=torch.tensor([[101, 7, 8], [101, 9, 102]]), **kw)),
           "groups": (lambda: LP.ProcessedGroupBeamState(2, 4, 300, 10, num_beam_groups=2, diversity_penalty=0.5),
                      lambda **kw: DA.ArgsGroupBeamState(2, 4, 300, 10, num_beam_groups=2, diversity_penalty=0.5, **kw)),
           "sample": (lambda: LP.ProcessedBeamSampleState(2, 4, 300, 10, N=2, seed=7),
                      lambda **kw: DA.ArgsBeamSampleState(2, 4, 300, 10, N=2, seed=7, **kw))}


@pytest.mark.parametrize("cls,N", [("beam", 1), ("beam", 3), ("groups", 1), ("groups", 3), ("sample", 1)])
def test_defaults_equal_the_existing_oracles(cls, N):
    """length_penalty 1, early_stopping off and no bad words: every step and the N-best finalisation are the existing oracle's (beam
    sampling returns one hypothesis per search)."""
    base, args = _STATES[cls]
    a, b = base(), args(length_penalty=1.0, early_stopping=False, bad_words_ids=None)
    for lg in _random_steps(a.B * a.K, 300, 10, 3):
        ra, rb = a.step(lg), b.step(lg)
        assert all(torch.equal(x, y) for x, y in zip(ra, rb))
        assert a.worst == b.worst and a.hyps == b.hyps
    fa, fb = finalize_nbest(a, N), finalize_nbest(b, N)
    assert all(torch.equal(x, y) for x, y in zip(fa, fb))


def test_hypothesis_scores_and_is_done():
    st = DA.ArgsGroupBeamState(1, 2, 50, 6, length_penalty=2.0)
    st._add(0, [5, 6], -3.0, 3)
    assert st.hyps[0] == [(-3.0 / 9.0, [5, 6])]
    assert not st._is_done(0, -1.0, 4)                   # one hypothesis, two beams
    st._add(0, [7], -1.0, 2)
    assert st.worst[0] == -3.0 / 9.0
    assert st._is_done(0, -6.0, 4) and not st._is_done(0, -5.0, 4)     # -3/9 >= -6/16, < -5/16
    zero = DA.ArgsGroupBeamState(1, 2, 50, 6, length_penalty=0.0)
    zero._add(0, [5], -3.0, 7)
    assert zero.hyps[0][0][0] == -3.0                    # no normalisation
    es = DA.ArgsGroupBeamState(1, 2, 50, 6, early_stopping=True)
    es._add(0, [5], -3.0, 2)
    assert not es._is_done(0, 0.0, 3)
    es._add(0, [6], -30.0, 2)
    assert es._is_done(0, 0.0, 3)                        # full heap: done whatever the scores
    odd = DA.ArgsGroupBeamState(1, 2, 50, 6, length_penalty=0.6)
    assert odd.length_penalty == float(np.float32(0.6)) and odd._denom(7) == 7.0 ** float(np.float32(0.6))
    for bad in (dict(length_penalty=float("inf")), dict(length_penalty=float("nan")), dict(early_stopping=2)):
        with pytest.raises(ValueError):
            DA.ArgsGroupBeamState(1, 2, 50, 6, **bad)


@pytest.fixture(scope="module")
def short_sd(tiny_sd):
    """Tiny weights whose hypotheses end early and at different lengths: the length penalty decides which one wins."""
    return _with_bias(tiny_sd, {R.EOS: 3.5})


def _tiny_batch(enc_cfg):
    return _with_question(history_batch(enc_cfg, 0, 3), A4["tiny"])


def test_the_arguments_change_results_on_the_tiny_model(tiny_cfgs, short_sd):
    enc_cfg, dec_cfg = tiny_cfgs
    b = _tiny_batch(enc_cfg)
    with torch.no_grad():
        out = {(lp, es): DA.group_beam_state(short_sd, enc_cfg, dec_cfg, b, 5, length_penalty=lp, early_stopping=es).finalize()
               for lp in (1.0, 2.0, -0.5) for es in (False, True)}
    base_ids, base_sc = out[(1.0, False)]
    assert not torch.equal(out[(2.0, False)][0], base_ids) and not torch.equal(out[(-0.5, False)][0], base_ids)
    assert any(not torch.equal(out[(lp, True)][0], out[(lp, False)][0]) for lp in (1.0, 2.0, -0.5))
    # a longer hypothesis wins more often with a larger length penalty
    length = lambda ids: float((ids != 0).sum())                            # noqa: E731
    assert length(out[(2.0, False)][0]) >= length(base_ids) >= length(out[(-0.5, False)][0])


# ---- GPU: tiny fp32 against the oracles -------------------------------------------------------------------------------
_ORACLE = {}
_SEED = 0x5EED
_WARP = dict(temperature=0.7, top_k=7, top_p=0.0)
MODES = {"beam3": dict(num_beams=3), "beam5": dict(num_beams=5), "nbest5": dict(num_beams=5, num_return_sequences=5),
         "groups": dict(num_beams=6, num_beam_groups=3, diversity_penalty=0.5),
         "beam_sample": dict(num_beams=3, do_sample=True, num_return_sequences=2, seed=_SEED, **_WARP)}


def _oracle(sd, enc_cfg, dec_cfg, b, mode, lp, es, n=0, prefix=None, row_offset=0, key_extra=()):
    key = (mode, lp, es, n, key_extra)
    if key not in _ORACLE:
        m = MODES[mode]
        with torch.no_grad():
            if mode == "beam_sample":
                _ORACLE[key] = DA.beam_sample(sd, enc_cfg, dec_cfg, b, m["num_beams"], m["num_return_sequences"], seed=_SEED, row_offset=row_offset,
                                              ngram_blocking_size=n, prefix=prefix, length_penalty=lp, early_stopping=es, **_WARP)
            else:
                st = DA.group_beam_state(sd, enc_cfg, dec_cfg, b, m["num_beams"], m.get("num_beam_groups", 1), m.get("diversity_penalty", 0.0),
                                         ngram_blocking_size=n, prefix=prefix, length_penalty=lp, early_stopping=es)
                _ORACLE[key] = finalize_nbest(copy.deepcopy(st), m.get("num_return_sequences", 1))
    return _ORACLE[key]


@pytest.fixture(scope="module")
def engines(tiny_cfgs, short_sd):
    from gst_visdial_b200 import _lib
    from test_logits_processors import _engine
    enc_cfg, dec_cfg = tiny_cfgs
    b = _tiny_batch(enc_cfg)
    es = {"separate_calls": _engine(enc_cfg, dec_cfg, short_sd, "fp32", b),
          "no_cuda_graph": _engine(enc_cfg, dec_cfg, short_sd, "fp32", b, flags=_lib.GSTVD_FLAG_NO_CUDA_GRAPH)}
    es["whole_round"] = es["separate_calls"]
    yield es, b
    for e in set(es.values()):
        e.close()


def _check_scores(mode, sc, ref_sc):
    # a last-bit difference of a logZ (the kernel's table-driven fp64 exp) stays in the fp32 beam sums, and len ** -lambda scales it
    # up with the score; beam sampling divides every step's scores by the temperature again: relative bounds, as in test_ragged_prefix
    tol = dict(rtol=2e-6, atol=1e-4) if mode == "beam_sample" else dict(rtol=2e-6, atol=1e-5)
    assert torch.allclose(sc.cpu().double(), ref_sc.double().view(-1), **tol), (sc, ref_sc)


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["separate_calls", "whole_round", "no_cuda_graph"])
@pytest.mark.parametrize("es", [False, True])
@pytest.mark.parametrize("lp", LAMBDAS)
@pytest.mark.parametrize("mode", sorted(MODES))
def test_tiny_fp32_matches_oracle(tiny_cfgs, short_sd, engines, mode, lp, es, path):
    from test_logits_processors import _run
    enc_cfg, dec_cfg = tiny_cfgs
    e, b = engines[0][path], engines[1]
    ref, ref_sc = _oracle(short_sd, enc_cfg, dec_cfg, b, mode, lp, es)
    ids, sc = _run(e, b, path, length_penalty=lp, early_stopping=es, **MODES[mode])
    assert torch.equal(ids.cpu(), ref), f"{ids.cpu().tolist()} vs {ref.tolist()}"
    _check_scores(mode, sc, ref_sc)


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["separate_calls", "whole_round", "no_cuda_graph"])
@pytest.mark.parametrize("lp,es", [(0.6, False), (2.0, True), (-0.5, False)])
def test_tiny_fp32_ragged_prefix_with_blocking(tiny_cfgs, short_sd, engines, lp, es, path):
    """Prefix lengths 1, 9 and 25 in one call with 4-gram question blocking: each image equals the oracle of that image alone."""
    from test_logits_processors import _run
    from test_ragged_prefix import TINY_LENS, per_image, tiny_prefix
    enc_cfg, dec_cfg = tiny_cfgs
    e, b = engines[0][path], engines[1]
    base, pre = tiny_prefix(enc_cfg)
    for mode in ("beam3", "nbest5", "groups", "beam_sample"):
        N = MODES[mode].get("num_return_sequences", 1)
        ids, sc = _run(e, b, path, ngram_blocking_size=4, prefix=pre, length_penalty=lp, early_stopping=es, **MODES[mode])
        ids, sc = ids.cpu().view(3, N, -1), sc.cpu().view(3, N)
        for i, Pb in enumerate(TINY_LENS):
            ref, ref_sc = _oracle(short_sd, enc_cfg, dec_cfg, per_image(b, i), mode, lp, es, n=4, prefix=base[i:i + 1, :Pb], row_offset=i,
                                  key_extra=("ragged", i))
            assert torch.equal(ids[i], ref), f"{mode}, image {i} (P_b={Pb}): {ids[i].tolist()} vs {ref.tolist()}"
            _check_scores(mode, sc[i], ref_sc)


@pytest.mark.gpu
def test_op_beam_entries_keep_the_hf_defaults(tiny_cfgs, tiny_sd):
    """The fp32 beam op entries score with length_penalty 1 and no early stopping, as the oracle of oracle/beam.py."""
    from oracle.beam import BeamState
    from test_logits_processors import _engine
    enc_cfg, dec_cfg = tiny_cfgs
    b = history_batch(enc_cfg, 0, 2)
    e = _engine(enc_cfg, dec_cfg, tiny_sd, "fp32", b)
    try:
        B, K, T, V = 2, 3, 8, enc_cfg.vocab_size
        st = BeamState(B, K, V, T)
        e.op_beam_begin(B, K, T)
        for lg in _random_steps(B * K, V, T, 5):
            bi, bt, _ = e.op_beam_step(lg.cuda())
            rbi, rbt, _ = st.step(lg)
            assert torch.equal(bi.cpu().long(), rbi) and torch.equal(bt.cpu().long(), rbt)
        ids, sc = e.op_beam_end(T)
        rids, rsc = st.finalize()
        assert torch.equal(ids.cpu(), rids) and torch.allclose(sc.cpu().double(), rsc, atol=1e-5)
    finally:
        e.close()


@pytest.mark.gpu
def test_graph_cache_recaptures_for_the_length_arguments(tiny_cfgs, short_sd, engines):
    from test_logits_processors import _run
    enc_cfg, dec_cfg = tiny_cfgs
    e, b = engines[0]["separate_calls"], engines[1]
    for lp, es in ((1.0, False), (2.0, False), (2.0, True), (-0.5, False), (1.0, False), (2.0, False)):
        ref, _ = _oracle(short_sd, enc_cfg, dec_cfg, b, "beam5", lp, es)
        ids, _ = _run(e, b, "separate_calls", length_penalty=lp, early_stopping=es, **MODES["beam5"])
        assert torch.equal(ids.cpu(), ref), (lp, es)


@pytest.mark.gpu
def test_rejections(tiny_cfgs, tiny_sd):
    from gst_visdial_b200._lib import GstvdError
    from test_logits_processors import _engine
    enc_cfg, dec_cfg = tiny_cfgs
    b = history_batch(enc_cfg, 0, 2)
    e = _engine(enc_cfg, dec_cfg, tiny_sd, "fp32", b)
    rnd = (b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"], b["enc_image_mask"])
    try:
        for mode in (dict(), dict(num_beams=3), dict(num_beams=3, do_sample=True, top_k=7)):
            for kw in (dict(length_penalty=float("inf")), dict(length_penalty=float("nan")), dict(length_penalty=-float("inf")),
                       dict(early_stopping=2), dict(early_stopping=-1)):
                with pytest.raises(GstvdError) as ei:
                    e.generate(2, **mode, **kw)
                assert ei.value.status == -1, kw
                with pytest.raises(GstvdError) as ei:
                    e.round(*rnd, **mode, **kw)
                assert ei.value.status == -1, kw
    finally:
        e.close()


# ---- GPU: full config, bf16 -------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_full_bf16_beam_arguments(full_cfgs, full_sd):
    """Teacher-style beam-5 with length_penalty / early_stopping: the launch count is that of the default call (1857), the defaults
    passed explicitly give the same bits as the call without them, and the returned scores are the penalised ones (score * len ** lp
    is the same fp32 sum whatever lp ranks by: checked on the hypothesis the two calls share)."""
    from test_logits_processors import _engine, _run
    enc_cfg, dec_cfg = full_cfgs
    b = history_batch(enc_cfg, 0, 4)
    e = _engine(enc_cfg, dec_cfg, full_sd, "bf16", b)
    try:
        ids0, sc0 = _run(e, b, "separate_calls", num_beams=5)
        ids1, sc1 = _run(e, b, "separate_calls", num_beams=5, length_penalty=1.0, early_stopping=False, bad_words_ids=None)
        assert torch.equal(ids0, ids1) and torch.equal(sc0, sc1)
        for kw in (dict(length_penalty=1.5), dict(early_stopping=True), dict(length_penalty=0.0, early_stopping=True)):
            before = e.launch_count
            ids, sc = _run(e, b, "separate_calls", num_beams=5, **kw)
            torch.cuda.synchronize()
            assert e.launch_count - before == 1857, kw
            lp = kw.get("length_penalty", 1.0)
            for r in range(4):
                if torch.equal(ids[r], ids0[r]):
                    n = int((ids0[r] != 0).sum()) - int((ids0[r] == R.EOS).any())    # generated tokens without the closing [SEP]
                    length = 1 + n
                    assert math.isclose(float(sc[r]) * length ** lp, float(sc0[r]) * length, rel_tol=1e-5, abs_tol=1e-5), (kw, r)
        ids_r, _ = _run(e, b, "whole_round", num_beams=5, length_penalty=1.5)
        ids_s, _ = _run(e, b, "separate_calls", num_beams=5, length_penalty=1.5)
        assert torch.equal(ids_r, ids_s)
    finally:
        e.close()
