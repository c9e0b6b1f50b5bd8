"""Decoder prefixes of different lengths in one decode call (include/gstvd.h gstvd_generate: a negative id ends an image's prefix).

Image b of a ragged call continues from prefix[b, :P_b] and must return exactly what a call holding image b alone with that prefix
returns, in every decode mode.  The oracle is the existing per-image one, run on image b alone with prefix[b, :P_b] and row_offset = b.
CPU: the Python layer rejects a row that starts with a negative id and passes every other prefix through unchanged.
GPU, fp32: greedy (with and without 4-gram blocking) equals the restatement per image; beam search, N-best, beam groups and beam
sampling, with and without the logits processors, equal their oracles per image on every call path; top-k sampling equals the uniform
call at each image's length.  bf16: padding columns are ignored bit for bit, a ragged batch agrees across call paths and with the
uniform call at each length, and launches as many kernels as a uniform call.  Kernel level: the self-attention kernels and the
ancestry update with per-image P0 against the fp64 reference / a Python model of the update.
"""
import copy
import types

import pytest
import torch

from helpers import R, history_batch
from oracle import processors as LP
from oracle.beam_nbest import finalize_nbest
from test_candidates import _sub
from test_decoder_prefix import A4, _GREEDY, _greedy_ref, _prefixes, _with_bias, _with_question

# P_b per image: [CLS] only, a 4-gram key across the prefix / output boundary, and 25 tokens (42 cached positions, the 64-position
# kernels) next to the short rows
TINY_LENS = (1, 9, 25)
TINY_P = 25


def ragged(base, lens, fill=-1):
    """base [B, P] with the columns of row b from lens[b] on set to negative ids (a different one per row)."""
    p = base.clone()
    for b, n in enumerate(lens):
        p[b, n:] = fill - b
    return p


def tiny_prefix(enc_cfg, B=3, P=TINY_P, lens=TINY_LENS):
    """A ragged [B, P] tiny prefix: row 1 ends with the first two tokens of the history 4-gram (its key spans the boundary at the
    first step) and repeats a token pair inside its prefix (repetition penalty / no_repeat_ngram_size act on the prefix)."""
    a, b4, _, _ = A4["tiny"]
    base = _prefixes(B, P, enc_cfg.vocab_size)
    n1 = lens[1]
    base[1, n1 - 2:n1] = torch.tensor([a, b4])
    base[1, 1:5] = torch.tensor([300, 301, 300, 301])
    return base, ragged(base, lens)


def per_image(b, i):
    return _sub(b, i, i + 1)


# ---- CPU -----------------------------------------------------------------------------------------------------------
def test_python_layer_checks_the_first_column():
    from gst_visdial_b200.engine import Engine
    stub = types.SimpleNamespace(_dev=lambda t, dtype: t)
    base = torch.tensor([[101, 7, 8], [101, 9, -1], [5, -1, -1]])
    pre, P = Engine._prefix(stub, base, 3)
    assert pre is base and P == 3                             # ragged rows pass through unchanged
    plain = torch.tensor([[101, 7], [101, 9]])
    pre, P = Engine._prefix(stub, plain, 2)
    assert pre is plain and P == 2
    assert Engine._prefix(stub, None, 2) == (None, 1)
    bad = base.clone()
    bad[1, 0] = -1
    with pytest.raises(ValueError, match="row 1"):
        Engine._prefix(stub, bad, 3)
    with pytest.raises(ValueError):
        Engine._prefix(stub, torch.tensor([[-5]]), 1)


# ---- GPU: fp32 greedy ----------------------------------------------------------------------------------------------
def _engine(enc_cfg, dec_cfg, sd, dtype, b, flags=0):
    from test_logits_processors import _engine as make
    return make(enc_cfg, dec_cfg, sd, dtype, b, flags)


@pytest.mark.gpu
@pytest.mark.parametrize("size", ["tiny", "full"])
def test_fp32_greedy_matches_restatement_per_image(size, tiny_cfgs, tiny_sd, full_cfgs, full_sd):
    enc_cfg, dec_cfg = tiny_cfgs if size == "tiny" else full_cfgs
    base_sd = tiny_sd if size == "tiny" else full_sd
    a, b4, c, d = A4[size]
    lens = TINY_LENS if size == "tiny" else (25, 1, 8)
    B, P = 3, 25
    b = _with_question(history_batch(enc_cfg, 0, B), A4[size])
    base = _prefixes(B, P, enc_cfg.vocab_size)
    i8 = lens.index(8) if 8 in lens else 1
    base[i8, lens[i8] - 3:lens[i8]] = torch.tensor([a, b4, c])     # without blocking the first step completes the history 4-gram
    pre = ragged(base, lens)
    sd = _with_bias(base_sd, {d: 30.0})
    e = _engine(enc_cfg, dec_cfg, sd, "fp32", b)
    try:
        for n in (0, 4):
            got = e.generate(B, num_beams=1, **_GREEDY, ngram_blocking_size=n, prefix=pre, hist_ids=b["enc_input_ids"],
                             hist_segments=b["enc_segments"]).cpu()
            for i in range(B):
                ref = _greedy_ref(sd, enc_cfg, dec_cfg, per_image(b, i), base[i:i + 1, :lens[i]], n=n)
                assert torch.equal(got[i:i + 1], ref), f"n={n}, image {i} (P_b={lens[i]}): {got[i].tolist()} vs {ref[0].tolist()}"
                if i == i8:
                    assert (ref[0, 0] == d) == (n == 0), "precondition: only blocking stops the 4-gram across the boundary"
    finally:
        e.close()


# ---- GPU: fp32 beam modes against the per-image oracles -------------------------------------------------------------
# min_length 12: [SEP] is allowed from the first step for the 25-token prefix and banned for the 1- and 9-token prefixes
PROCS_ON = dict(repetition_penalty=1.3, no_repeat_ngram_size=3, min_length=12)
_BS_WARP = dict(temperature=0.7, top_k=7, top_p=0.0)
_SEED = 0x5EED
_ORACLE = {}


def _modes(K):
    """(name, generate kwargs) of the beam modes run at beam width K; groups need K % 3 == 0, so K = 5 runs them at 6 beams."""
    return [("beam", dict(num_beams=K)), ("nbest", dict(num_beams=K, num_return_sequences=2)),
            ("groups", dict(num_beams=3 if K == 3 else 6, num_beam_groups=3, diversity_penalty=0.5)),
            ("beam_sample", dict(num_beams=4, num_return_sequences=2, do_sample=True, seed=_SEED, **_BS_WARP))]


def _oracle_image(sd, enc_cfg, dec_cfg, b, i, prefix, name, kw, n, procs):
    """(ids [N, 18], scores [N]) of image i alone with its own prefix, from the existing oracles (row_offset = i)."""
    key = (name, tuple(sorted((k, v) for k, v in kw.items())), n, procs is not None, i)
    if key not in _ORACLE:
        bi = per_image(b, i)
        with torch.no_grad():
            if name == "beam_sample":
                _ORACLE[key] = LP.beam_sample(sd, enc_cfg, dec_cfg, bi, kw["num_beams"], kw["num_return_sequences"], seed=_SEED, row_offset=i,
                                              ngram_blocking_size=n, prefix=prefix, processors=procs, **_BS_WARP)
            else:
                st = LP.group_beam_state(sd, enc_cfg, dec_cfg, bi, kw["num_beams"], kw.get("num_beam_groups", 1), kw.get("diversity_penalty", 0.0),
                                         ngram_blocking_size=n, prefix=prefix, processors=procs)
                _ORACLE[key] = finalize_nbest(copy.deepcopy(st), kw.get("num_return_sequences", 1))
    return _ORACLE[key]


@pytest.fixture(scope="module")
def tiny_engines(tiny_cfgs, tiny_sd):
    from gst_visdial_b200 import _lib
    enc_cfg, dec_cfg = tiny_cfgs
    sd = _with_bias(tiny_sd, {R.EOS: 3.5, A4["tiny"][3]: 3.0})     # hypotheses end early; the history 4-gram is attractive
    b = _with_question(history_batch(enc_cfg, 0, 3), A4["tiny"])
    es = {"separate_calls": _engine(enc_cfg, dec_cfg, sd, "fp32", b),
          "no_cuda_graph": _engine(enc_cfg, dec_cfg, sd, "fp32", b, flags=_lib.GSTVD_FLAG_NO_CUDA_GRAPH)}
    es["whole_round"] = es["separate_calls"]
    yield es, b, sd
    for e in set(es.values()):
        e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["separate_calls", "whole_round", "no_cuda_graph"])
@pytest.mark.parametrize("procs", ["off", "on"])
@pytest.mark.parametrize("n", [0, 4])
@pytest.mark.parametrize("K", [3, 5])
def test_tiny_fp32_ragged_beams_match_per_image_oracles(tiny_cfgs, tiny_engines, K, n, procs, path):
    from test_logits_processors import _run
    enc_cfg, dec_cfg = tiny_cfgs
    es, b, sd = tiny_engines
    base, pre = tiny_prefix(enc_cfg)
    p = PROCS_ON if procs == "on" else None
    for name, kw in _modes(K):
        N = kw.get("num_return_sequences", 1)
        ids, sc = _run(es[path], b, path, ngram_blocking_size=n, prefix=pre, **kw, **(p or {}))
        ids, sc = ids.cpu().view(3, N, -1), sc.cpu().view(3, N)
        for i, Pb in enumerate(TINY_LENS):
            ref, ref_sc = _oracle_image(sd, enc_cfg, dec_cfg, b, i, base[i:i + 1, :Pb], name, kw, n, p)
            what = f"{name}, image {i} (P_b={Pb})"
            assert torch.equal(ids[i], ref), f"{what}: {ids[i].tolist()} vs {ref.tolist()}"
            assert torch.allclose(sc[i].double(), ref_sc.double().view(-1), rtol=2e-6, atol=1e-4), f"{what}: {sc[i]} vs {ref_sc}"
        if procs == "on" and name == "beam":
            # min_length at work per row: no [SEP] in the first step of the short rows, and the long row closes early
            first_sep = [int((r == R.EOS).nonzero()[0]) if (r == R.EOS).any() else 18 for r in ids[:, 0]]
            assert first_sep[0] >= 12 - 1 and first_sep[1] >= 12 - 9, first_sep


@pytest.mark.gpu
def test_tiny_fp32_invalid_row_leaves_the_others_exact(tiny_cfgs, tiny_engines):
    """A row that starts with a negative id is invalid input with unspecified output; the call still completes and every other
    image decodes exactly as alone."""
    enc_cfg, dec_cfg = tiny_cfgs
    es, b, sd = tiny_engines
    base, pre = tiny_prefix(enc_cfg)
    bad = pre.clone()
    bad[0, :] = -7
    e = es["separate_calls"]
    hist = dict(hist_ids=b["enc_input_ids"], hist_segments=b["enc_segments"])
    for kw in (dict(num_beams=3, ngram_blocking_size=4, **PROCS_ON), dict(num_beams=1, temperature=0.7, top_k=7, seed=3, ngram_blocking_size=4)):
        got = e.generate(3, prefix=bad.to(e.device), **kw, **hist).cpu()      # a device tensor is not checked on the host
        want = e.generate(3, prefix=pre, **kw, **hist).cpu()
        assert torch.equal(got[1:], want[1:])


# ---- GPU: fp32 sampling against the uniform call at each length ------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("path", ["separate_calls", "whole_round"])
@pytest.mark.parametrize("N", [1, 3])
def test_tiny_fp32_ragged_sampling_equals_uniform_calls(tiny_cfgs, tiny_engines, N, path):
    from test_logits_processors import _run
    enc_cfg, dec_cfg = tiny_cfgs
    es, b, sd = tiny_engines
    base, pre = tiny_prefix(enc_cfg)
    for extra in (dict(ngram_blocking_size=4), dict(ngram_blocking_size=0, **PROCS_ON)):
        kw = dict(num_beams=1, temperature=0.7, top_k=7, top_p=0.0, seed=91, num_return_sequences=N, **extra)
        got = _run(es[path], b, path, prefix=pre, **kw)[0].cpu().view(3, N, -1)
        for i, Pb in enumerate(TINY_LENS):
            uni = _run(es[path], b, path, prefix=base[:, :Pb].contiguous(), **kw)[0].cpu().view(3, N, -1)
            assert torch.equal(got[i], uni[i]), f"{extra}, image {i} (P_b={Pb}): {got[i].tolist()} vs {uni[i].tolist()}"


# ---- GPU: bf16 product path -----------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_full_bf16_ragged_prefixes(full_cfgs, full_sd):
    from gst_visdial_b200 import _lib
    from test_logits_processors import _run
    enc_cfg, dec_cfg = full_cfgs
    B, P = 64, 25
    b = history_batch(enc_cfg, 0, B)
    base = _prefixes(B, P, enc_cfg.vocab_size)
    lens = torch.randint(1, P + 1, (B,), generator=torch.Generator().manual_seed(4)).tolist()
    lens[:3] = [1, P, 9]
    pre = ragged(base, lens)
    modes = {"beam": dict(num_beams=5, **_GREEDY), "sample": dict(num_beams=1, temperature=0.7, top_k=7, top_p=0.0, seed=11)}
    e = _engine(enc_cfg, dec_cfg, full_sd, "bf16", b)
    eager = _engine(enc_cfg, dec_cfg, full_sd, "bf16", b, flags=_lib.GSTVD_FLAG_NO_CUDA_GRAPH)
    try:
        for m, mk in modes.items():
            kw = dict(mk, ngram_blocking_size=4)
            # 1. every image of P' = 10 tokens, padded with negative ids to P: bit-identical ids and scores to the [B, P'] call
            short = base[:, :10].contiguous()
            want = _run(e, b, "separate_calls", prefix=short, **kw)
            got = _run(e, b, "separate_calls", prefix=ragged(base, [10] * B), **kw)
            assert torch.equal(got[0], want[0]), f"{m}: padding columns change the ids"
            if m == "beam":
                assert torch.equal(got[1], want[1]), f"{m}: padding columns change the scores"
            # 2. a ragged batch: the same ids on every path and on repeated calls, as many launches as a uniform [B, P] call
            l0 = e.launch_count
            ids = _run(e, b, "separate_calls", prefix=pre, **kw)[0].cpu()
            l1 = e.launch_count
            _run(e, b, "separate_calls", prefix=base, **kw)
            l2 = e.launch_count
            assert l1 - l0 == l2 - l1, f"{m}: a ragged call launches {l1 - l0} kernels, a uniform one {l2 - l1}"
            assert torch.equal(_run(e, b, "separate_calls", prefix=pre, **kw)[0].cpu(), ids), f"{m}: repeated calls differ"
            assert torch.equal(_run(e, b, "whole_round", prefix=pre, **kw)[0].cpu(), ids), f"{m}: whole-round graph differs"
            assert torch.equal(_run(eager, b, "separate_calls", prefix=pre, **kw)[0].cpu(), ids), f"{m}: eager decode differs"
            # 3. each image agrees with the uniform call at its own length.  The prefill runs over P - 1 columns instead of P_b - 1, but
            # its GEMM and attention rows do not depend on the other rows or on later columns, and the decode step's per-row
            # arithmetic does not depend on the padded width: identity is expected.
            for Pb in sorted(set(lens)):
                uni = _run(e, b, "separate_calls", prefix=base[:, :Pb].contiguous(), **kw)[0].cpu()
                rows = [i for i, n in enumerate(lens) if n == Pb]
                assert torch.equal(ids[rows], uni[rows]), f"{m}: images {rows} (P_b={Pb}) differ from the uniform call"
    finally:
        e.close()
        eager.close()


# ---- GPU: kernel level ----------------------------------------------------------------------------------------------
def _ragged_self_inputs(B, K, heads, D, T, p0s, step, seed, dtype, with_anc):
    """qkv, cache with NaN at and past every image's own new position (p0s[b] + step), ancestry with stale entries from there on."""
    from test_gpu_decode_attention import _round
    g = torch.Generator().manual_seed(seed)
    H = heads * D
    qkv = torch.cat([torch.randn(B * K, H, generator=g), torch.randn(B * K, H, generator=g), torch.rand(B * K, H, generator=g) * 2 - 1], 1)
    cache = torch.stack([torch.randn(B, T, K, H, generator=g), torch.rand(B, T, K, H, generator=g) * 2 - 1])
    anc = None
    if with_anc:
        W = 32 if T <= 32 else 64
        anc = torch.randint(0, K, (B * K, W), generator=g)
    for b, p0 in enumerate(p0s):
        cache[:, b, p0 + step:] = float("nan")
        if anc is not None:
            anc[b * K:(b + 1) * K, p0 + step:] = torch.randint(K, 256, (K, anc.shape[1] - p0 - step), generator=g)
    return _round(qkv, dtype), _round(cache, dtype), None if anc is None else anc.to(torch.uint8)


@pytest.fixture(scope="module")
def attn_eng(full_cfgs):
    from gst_visdial_b200.engine import Engine
    enc_cfg, dec_cfg = full_cfgs
    e = Engine(enc_cfg, dec_cfg, device=0, dtype="bf16", max_batch=8, max_beams=5)
    yield e
    e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,dtype,D,with_anc", [("v2", "bf16", 64, False), ("v2", "bf16", 64, True), ("first", "bf16", 64, False),
                                                      ("first", "bf16", 128, False), ("first", "fp32", 64, False), ("first", "fp32", 128, False)])
@pytest.mark.parametrize("T,P0,step", [(20, 12, 0), (21, 12, 5), (33, 25, 7), (43, 25, 0), (64, 46, 17)])
def test_self_attention_per_image_p0(attn_eng, kernel, dtype, D, with_anc, T, P0, step):
    from test_gpu_decode_attention import check_close, ref_self_attn, ref_self_cache, same_bits
    B, K, heads = 4, (8 if with_anc else 5), 768 // D
    p0s = [P0, 0, P0 // 2, 1]
    qkv, cache, anc = _ragged_self_inputs(B, K, heads, D, T, p0s, step, T * 100 + step + D, dtype, with_anc)
    for step_known in (True, False):
        y, c = attn_eng.op_dec_self_attn(qkv, cache, heads, P0=P0, step=step, step_known=step_known, anc=anc, kernel=kernel, dtype=dtype,
                                         p0s=torch.tensor(p0s, dtype=torch.int32))
        y, c = y.cpu(), c.cpu()
        for b, p0 in enumerate(p0s):
            rows = slice(b * K, (b + 1) * K)
            exp = ref_self_cache(qkv[rows], cache[:, b:b + 1], None, 1, K, p0, step)
            ref = ref_self_attn(qkv[rows], exp, None if anc is None else anc[rows], 1, K, heads, p0, step)
            what = f"{kernel}/{dtype} D={D} anc={with_anc} T={T} P0={P0} step={step} step_known={step_known} image {b} (P0_b={p0})"
            check_close(y[rows], ref, kernel, dtype, what)
            assert same_bits(c[:, b:b + 1], exp), f"{what}: the cache differs from the input + appended k/v"


@pytest.mark.gpu
@pytest.mark.parametrize("T,P0", [(30, 12), (64, 40)])
def test_anc_update_per_image_p0(attn_eng, T, P0):
    B, K = 4, 5
    W = 32 if T <= 32 else 64
    g = torch.Generator().manual_seed(T)
    p0s = [P0, 0, P0 // 3, 1]
    anc = torch.randint(0, 256, (B * K, W), generator=g).to(torch.uint8)
    for step in range(T - P0):
        parent = torch.randint(0, K, (B, K), generator=g)
        got = attn_eng.op_anc_update(anc, parent, T, P0, step, p0s=torch.tensor(p0s, dtype=torch.int32)).cpu()
        want = anc.view(B, K, W).clone()
        for b, p0 in enumerate(p0s):
            pos = p0 + step
            want[b, :, :pos] = anc.view(B, K, W)[b, parent[b], :pos]
            want[b, :, pos] = parent[b].to(torch.uint8)
        assert torch.equal(got, want.view(B * K, W)), f"step {step}"
        anc = got
