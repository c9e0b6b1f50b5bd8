"""GPU: the whole hot path through the reference-shaped module API / C ABI against the oracle and the golden vectors.

Tolerances (BASELINE.json north_star): fp32 logits <= 1e-3 max abs, greedy / beam ids identical in fp32;
bf16: 2e-2 relative, defined here as rms(delta) / rms(reference) over the logits of valid positions.
"""
import os

import numpy as np
import pytest
import torch

from helpers import R, history_batch, load_golden, max_abs, rel_rms
from oracle import beam as OB

pytestmark = pytest.mark.gpu

FP32_LOGIT_TOL = 1e-3
BF16_REL_TOL = 2e-2


def _params(enc_path, dec_path, dtype, model="enc_dec_a", mode="cc12m_gen", **kw):
    p = {"model_enc_config": enc_path, "model_dec_config": dec_path, "gpu_ids": [0], "model": model, "mode": mode,
         "compute_dtype": dtype, "engine_max_batch": 8, "engine_max_beams": 5}
    p.update(kw)
    return p


def _build_model(enc_path, dec_path, sd, dtype, **kw):
    from gst_visdial_b200.models.visual_dialog_decoder import VisualDialogDecoder
    from gst_visdial_b200.models.visual_dialog_encoder import VisualDialogEncoder
    from gst_visdial_b200.models.visual_dialog_model import EncoderDecoderModel
    params = _params(enc_path, dec_path, dtype, **kw)
    enc, dec = VisualDialogEncoder(params), VisualDialogDecoder(params)
    dec.decoder.bert.embeddings = enc.bert_pretrained.bert.embeddings          # generate.py:65
    model = EncoderDecoderModel(params, enc, dec)
    model = torch.nn.DataParallel(model, [0])                                  # generate.py:67
    model.module.load_state_dict(sd)                                           # generate.py:69
    model.to("cuda:0").eval()
    return model, params


def _call(model, b, dec_ids=None, **kw):
    dev = "cuda:0"
    dec = b["dec_input_ids"].clone() if dec_ids is None else dec_ids
    dec = dec.to(dev)
    out = model(enc_image_features=b["enc_image_feat"].to(dev), enc_image_spatials=b["enc_image_loc"].to(dev),
                enc_image_mask=b["enc_image_mask"].to(dev), enc_image_target=None, enc_image_label=None,
                enc_next_sentence_labels=None, enc_input_ids=b["enc_input_ids"].to(dev), enc_segments=b["enc_segments"].to(dev),
                enc_sep_indices=None, enc_mlm_labels=None, enc_attention_mask=b["enc_att_mask"].to(dev), dec_input_ids=dec,
                dec_attention_mask=(dec != 0).float(), **kw)
    return out, dec


@pytest.fixture(scope="module")
def tiny_fp32(tiny_sd):
    from gst_visdial_b200 import weights as W
    return _build_model(W.TINY_ENC_CONFIG, W.TINY_DEC_CONFIG, tiny_sd, "fp32")


@pytest.fixture(scope="module")
def tiny_bf16(tiny_sd):
    from gst_visdial_b200 import weights as W
    return _build_model(W.TINY_ENC_CONFIG, W.TINY_DEC_CONFIG, tiny_sd, "bf16")


def test_tiny_fp32_encoder_matches_golden(tiny_fp32, tiny_cfgs, golden_dir):
    model, _ = tiny_fp32
    g = load_golden(golden_dir, "tiny_b3")
    b = history_batch(tiny_cfgs[0], 0, 3)
    eng = model.module._engine(torch.device("cuda:0"))
    out = eng.encode(b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"],
                     b["enc_image_mask"], want_t=True, want_v=True, want_fused=True, want_nsp=True)
    assert max_abs(out["seq_v"].cpu(), torch.from_numpy(g["seq_v"])) < 1e-3
    assert max_abs(out["seq_t"].cpu(), torch.from_numpy(g["seq_t"])) < 1e-3
    assert max_abs(out["fused"].cpu(), torch.from_numpy(g["fused"])) < 1e-3
    assert max_abs(out["nsp"].cpu(), torch.from_numpy(g["nsp"])) < 1e-3
    assert torch.equal(out["fused_mask"].cpu(), torch.cat((b["enc_image_mask"], b["enc_att_mask"]), 1))
    # the wrapper returns the reference's 7-tuple
    tup = model.module.encoder(b["enc_input_ids"].cuda(), b["enc_image_feat"].cuda(), b["enc_image_loc"].cuda(),
                               token_type_ids=b["enc_segments"].cuda(), attention_mask=b["enc_att_mask"].cuda(),
                               image_attention_mask=b["enc_image_mask"].cuda())
    assert len(tup) == 7 and tup[0] is None and max_abs(tup[5].cpu(), torch.from_numpy(g["seq_t"])) < 1e-3


def test_tiny_fp32_greedy_ngram_score_match_golden(tiny_fp32, tiny_cfgs, golden_dir):
    model, params = tiny_fp32
    g = load_golden(golden_dir, "tiny_b3")
    b = history_batch(tiny_cfgs[0], 0, 3)
    seq, _ = _call(model, b, temperature=1.0, top_k=1, top_p=0.0, ngram_blocking_size=0)
    assert np.array_equal(seq.cpu().numpy(), g["greedy_ids"]), f"{seq.cpu().numpy()} vs {g['greedy_ids']}"
    seq_ng, _ = _call(model, b, temperature=0.7, top_k=1, top_p=0.0, ngram_blocking_size=4)
    assert np.array_equal(seq_ng.cpu().numpy(), g["greedy_ng4_ids"])
    # teacher-forced logits along the greedy path, then the perplexity pass of generate.py:183-209
    params["mode"] = "train"
    try:
        dec_in = torch.cat((b["dec_input_ids"], torch.from_numpy(g["greedy_ids"])[:, :-1]), 1)
        (loss, logits), _ = _call(model, b, dec_ids=dec_in, loss_reduction=False)
        assert max_abs(logits.cpu(), torch.from_numpy(g["greedy_logits"])) < FP32_LOGIT_TOL
        ans = torch.from_numpy(g["greedy_ids"]).clone()
        (loss, logits), ans_dev = _call(model, b, dec_ids=ans, loss_reduction=False)
        assert loss.shape == (3 * 18,)
        assert max_abs(loss.cpu().reshape(3, 18), torch.from_numpy(g["score_loss"])) < FP32_LOGIT_TOL
        assert max_abs(logits.cpu(), torch.from_numpy(g["score_logits"])) < FP32_LOGIT_TOL
        assert not (ans_dev == 102).any(), "dec_input_ids must be modified in place like the reference does"
        ans_len = (ans_dev != 0).sum(-1)
        ppl = torch.exp(loss.reshape(3, 18).sum(-1) / ans_len)
        assert np.allclose(ppl.cpu().numpy(), g["score_ppl"], rtol=2e-3)
        # mean reduction + reuse of the resident encoder state
        (loss_m, _), _ = _call(model, b, dec_ids=torch.from_numpy(g["greedy_ids"]).clone(), loss_reduction=True, reuse_encoder=True)
        sl = torch.from_numpy(g["score_loss"])
        assert abs(loss_m.item() - (sl.sum() / (sl != 0).sum()).item()) < 1e-3
    finally:
        params["mode"] = "cc12m_gen"


def test_tiny_fp32_beam_matches_oracle(tiny_fp32, tiny_cfgs, tiny_sd):
    model, _ = tiny_fp32
    enc_cfg, dec_cfg = tiny_cfgs
    b = history_batch(enc_cfg, 0, 3)
    with torch.no_grad():
        ref_seq, ref_sc = OB.beam_search(tiny_sd, enc_cfg, dec_cfg, b, num_beams=5)
    seq, _ = _call(model, b, temperature=1.0, top_k=1, top_p=0.0, ngram_blocking_size=0, num_beams=5)
    assert torch.equal(seq.cpu(), ref_seq), f"{seq.cpu()} vs {ref_seq}"
    eng = model.module._engine(torch.device("cuda:0"))
    seq2, sc2 = eng.generate(3, num_beams=5, want_scores=True)
    assert torch.equal(seq2.cpu(), ref_seq) and torch.allclose(sc2.cpu().double(), ref_sc, atol=1e-4)


def test_tiny_eos_handling(tiny_cfgs, tiny_sd):
    """Make [SEP] likely (large lm_head bias) so that EOS->PAD in the prefix, PAD-after-EOS and beam hypotheses are exercised."""
    from gst_visdial_b200 import weights as W
    enc_cfg, dec_cfg = tiny_cfgs
    sd = dict(tiny_sd)
    bias = sd["decoder.decoder.lm_head.bias"].clone()
    bias[102] += 2.5
    sd["decoder.decoder.lm_head.bias"] = bias
    sd["decoder.decoder.lm_head.decoder.bias"] = bias
    model, _ = _build_model(W.TINY_ENC_CONFIG, W.TINY_DEC_CONFIG, sd, "fp32")
    b = history_batch(enc_cfg, 0, 3)
    with torch.no_grad():
        ref = R.generate_greedy_or_sample(sd, enc_cfg, dec_cfg, b, 1.0, 1, 0.0, 0)
        ref_beam, _ = OB.beam_search(sd, enc_cfg, dec_cfg, b, num_beams=3)
    assert (ref == 102).any(), "test needs an EOS in the greedy output; raise the bias"
    seq, _ = _call(model, b, temperature=1.0, top_k=1, top_p=0.0, ngram_blocking_size=0)
    assert torch.equal(seq.cpu(), ref)
    seqb, _ = _call(model, b, temperature=1.0, top_k=1, top_p=0.0, ngram_blocking_size=0, num_beams=3)
    assert torch.equal(seqb.cpu(), ref_beam)


def test_tiny_graph_equals_eager(tiny_cfgs, tiny_sd):
    from gst_visdial_b200 import _lib
    from gst_visdial_b200.engine import Engine
    enc_cfg, dec_cfg = tiny_cfgs
    b = history_batch(enc_cfg, 0, 3)
    outs = []
    for flags in (0, _lib.GSTVD_FLAG_NO_CUDA_GRAPH):
        e = Engine(enc_cfg, dec_cfg, dtype="fp32", max_batch=4, flags=flags)
        e.load_state_dict(tiny_sd)
        enc = e.encode(b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"], b["enc_image_mask"])
        e.prefill_cross(3, enc["Le"])
        o1 = e.generate(3, num_beams=5).cpu()
        o2 = e.generate(3, num_beams=1, top_k=1).cpu()
        o3 = e.generate(3, num_beams=5).cpu()          # replay of the cached graph
        assert torch.equal(o1, o3)
        assert e.launch_count > 0
        outs.append((o1, o2))
        e.close()
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])


def test_tiny_bf16_within_tolerance(tiny_bf16, tiny_cfgs, golden_dir):
    model, params = tiny_bf16
    g = load_golden(golden_dir, "tiny_b3")
    b = history_batch(tiny_cfgs[0], 0, 3)
    eng = model.module._engine(torch.device("cuda:0"))
    out = eng.encode(b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"],
                     b["enc_image_mask"], want_t=True, want_v=True, want_fused=True, want_nsp=True)
    valid = b["enc_att_mask"].bool()
    rt = rel_rms(out["seq_t"].cpu()[valid], torch.from_numpy(g["seq_t"])[valid])
    rv = rel_rms(out["seq_v"].cpu(), torch.from_numpy(g["seq_v"]))
    print(f"bf16 encoder rel rms: text {rt:.4f} image {rv:.4f}")
    assert rt < BF16_REL_TOL and rv < BF16_REL_TOL
    params["mode"] = "train"
    try:
        dec_in = torch.cat((b["dec_input_ids"], torch.from_numpy(g["greedy_ids"])[:, :-1]), 1)
        (loss, logits), _ = _call(model, b, dec_ids=dec_in, loss_reduction=False)
    finally:
        params["mode"] = "cc12m_gen"
    rl = rel_rms(logits.cpu(), torch.from_numpy(g["greedy_logits"]))
    print(f"bf16 greedy-path logits rel rms {rl:.4f}, max abs {max_abs(logits.cpu(), torch.from_numpy(g['greedy_logits'])):.4f}")
    assert rl < BF16_REL_TOL
    seq, _ = _call(model, b, temperature=1.0, top_k=1, top_p=0.0, ngram_blocking_size=0)
    agree = (seq.cpu().numpy() == g["greedy_ids"]).mean()
    print(f"bf16 greedy token agreement with fp32 reference: {agree:.3f}")
    assert seq.shape == (3, 18)


def test_tiny_sampling_runs_and_is_seeded(tiny_bf16, tiny_cfgs):
    model, _ = tiny_bf16
    b = history_batch(tiny_cfgs[0], 0, 3)
    a, _ = _call(model, b, temperature=0.7, top_k=7, top_p=0.0, ngram_blocking_size=4, seed=11)
    c, _ = _call(model, b, temperature=0.7, top_k=7, top_p=0.0, ngram_blocking_size=4, seed=11)
    d, _ = _call(model, b, temperature=0.7, top_k=7, top_p=0.0, ngram_blocking_size=4, seed=12)
    assert torch.equal(a, c) and a.shape == (3, 18) and a.dtype == torch.int64
    assert not torch.equal(a, d)


def test_enc_only_nsp(tiny_cfgs, tiny_sd, golden_dir):
    from gst_visdial_b200 import weights as W
    from gst_visdial_b200.models.visual_dialog_encoder import VisualDialogEncoder
    g = load_golden(golden_dir, "tiny_b3")
    params = _params(W.TINY_ENC_CONFIG, W.TINY_DEC_CONFIG, "fp32", model="enc_only_a", mode="vd_eval_val")
    enc = VisualDialogEncoder(params)
    enc.load_state_dict({k[len("encoder."):]: v for k, v in tiny_sd.items() if k.startswith("encoder.")})
    enc.to("cuda:0").eval()
    b = history_batch(tiny_cfgs[0], 0, 3)
    out = enc(b["enc_input_ids"].cuda(), b["enc_image_feat"].cuda(), b["enc_image_loc"].cuda(), token_type_ids=b["enc_segments"].cuda(),
              attention_mask=b["enc_att_mask"].cuda(), image_attention_mask=b["enc_image_mask"].cuda())
    assert out[5] is None and max_abs(out[3].cpu(), torch.from_numpy(g["nsp"])) < 1e-3


# ---- full-size model (config/bert_base_6layer_6conect_*.json) ---------------------------------------------------------
@pytest.fixture(scope="module")
def full_engines(full_cfgs, full_sd):
    from gst_visdial_b200.engine import Engine
    enc_cfg, dec_cfg = full_cfgs
    e32 = Engine(enc_cfg, dec_cfg, dtype="fp32", max_batch=4)
    e32.load_state_dict(full_sd)
    e16 = Engine(enc_cfg, dec_cfg, dtype="bf16", max_batch=4)
    e16.load_state_dict(full_sd)
    yield e32, e16
    e32.close(); e16.close()


def test_full_fp32_config1_matches_reference_golden(full_engines, full_cfgs, golden_dir):
    """BASELINE.json configs[0]: teacher enc_dec_a, greedy, batch 1, fp32 - token ids identical, logits <= 1e-3."""
    e32, _ = full_engines
    g = load_golden(golden_dir, "full_b1")
    b = history_batch(full_cfgs[0], 0, 1)
    out = e32.encode(b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"], b["enc_image_mask"],
                     want_t=True, want_v=True, want_fused=True, want_nsp=True)
    assert max_abs(out["seq_t"].cpu()[:, :48, :32], torch.from_numpy(g["seq_t_slice"])) < 1e-3
    assert max_abs(out["seq_v"].cpu()[:, :, :32], torch.from_numpy(g["seq_v_slice"])) < 1e-3
    assert max_abs(out["fused"].cpu()[:, :, :24], torch.from_numpy(g["fused_slice"])) < 1e-3
    assert max_abs(out["fused"].cpu().sum(-1), torch.from_numpy(g["fused_rowsum"])) < 2e-2
    assert max_abs(out["nsp"].cpu(), torch.from_numpy(g["nsp"])) < 1e-3
    e32.prefill_cross(1, out["Le"])
    seq = e32.generate(1, num_beams=1, top_k=1, temperature=1.0)
    assert np.array_equal(seq.cpu().numpy(), g["greedy_ids"]), f"{seq.cpu().numpy()} vs {g['greedy_ids']}"
    dec_in = torch.cat((b["dec_input_ids"], torch.from_numpy(g["greedy_ids"])[:, :-1]), 1).cuda()
    _, logits = e32.score(dec_in, None, labels=torch.zeros_like(dec_in), want_logits=True)
    lg = logits.cpu()
    assert max_abs(lg[:, :, :256], torch.from_numpy(g["greedy_logits_slice"])) < FP32_LOGIT_TOL
    assert max_abs(torch.logsumexp(lg, -1), torch.from_numpy(g["greedy_logits_lse"])) < FP32_LOGIT_TOL
    top = lg.topk(8, dim=-1)
    assert np.array_equal(top.indices.numpy(), g["greedy_logits_top_idx"])
    ans = torch.from_numpy(g["greedy_ids"]).clone().cuda()
    loss, _ = e32.score(ans, (ans != 0).float())
    assert max_abs(loss.cpu(), torch.from_numpy(g["score_loss"])) < FP32_LOGIT_TOL


def test_full_bf16_vs_fp32(full_engines, full_cfgs, golden_dir):
    e32, e16 = full_engines
    g = load_golden(golden_dir, "full_b1")
    b = history_batch(full_cfgs[0], 0, 3)
    outs = []
    for e in (e32, e16):
        o = e.encode(b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"], b["enc_image_mask"],
                     want_t=True, want_v=True)
        e.prefill_cross(3, o["Le"])
        dec_in = torch.cat((b["dec_input_ids"].repeat(1, 1), torch.from_numpy(g["greedy_ids"]).repeat(3, 1)[:, :-1]), 1).cuda()
        _, lg = e.score(dec_in, None, labels=torch.zeros_like(dec_in), want_logits=True)
        outs.append((o["seq_t"].cpu(), o["seq_v"].cpu(), lg.cpu()))
    valid = b["enc_att_mask"].bool()
    rt = rel_rms(outs[1][0][valid], outs[0][0][valid]); rv = rel_rms(outs[1][1], outs[0][1]); rl = rel_rms(outs[1][2], outs[0][2])
    print(f"full model bf16 vs fp32: text {rt:.4f} image {rv:.4f} logits {rl:.4f} (max abs {max_abs(outs[1][2], outs[0][2]):.4f})")
    assert rt < BF16_REL_TOL and rv < BF16_REL_TOL and rl < BF16_REL_TOL
    s16 = e16.generate(3, num_beams=5)
    s32 = e32.generate(3, num_beams=5)
    print("beam-5 token agreement bf16 vs fp32:", (s16 == s32).float().mean().item())
    assert s16.shape == (3, 18)


@pytest.mark.parametrize("hist", [256, 140])
def test_full_cached_decode_agrees_with_teacher_forced_pass(full_engines, full_cfgs, hist):
    """KV-cached decode steps (decode-step attention kernels over the self / cross caches, Le up to 293) against the
    teacher-forced pass over the same tokens (different kernels, same weights): the argmax of the teacher-forced logits
    reproduces the greedy tokens.  Full-length histories exercise every key group / TMA box of the cross-attention."""
    e32, e16 = full_engines
    enc_cfg = full_cfgs[0]
    B = 3
    b = history_batch(enc_cfg, 0, B)
    g = torch.Generator().manual_seed(hist)
    ids = b["enc_input_ids"]
    for i in range(B):
        n = int((ids[i] != 0).sum())
        ids[i, n:hist] = torch.randint(1000, enc_cfg.vocab_size, (hist - n,), generator=g)
    b["enc_att_mask"] = (ids != 0).float()
    for e, need in ((e32, 0.98), (e16, 0.75)):           # bf16: near-tied logits of a random-weight model may flip the argmax
        o = e.encode(ids, b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"], b["enc_image_mask"])
        e.prefill_cross(B, o["Le"])
        out = e.generate(B, num_beams=1, top_k=1)
        dec_in = torch.cat((torch.full((B, 1), 101, dtype=torch.int64, device=out.device), out[:, :-1]), 1).contiguous()
        _, lg = e.score(dec_in, None, labels=torch.zeros_like(dec_in), want_logits=True)
        assert torch.isfinite(lg).all()
        agree = (lg.argmax(-1) == out).float().mean().item()
        top3 = (lg.topk(3, -1).indices == out.unsqueeze(-1)).any(-1).float().mean().item()
        assert top3 >= 0.95, f"generated tokens inside the teacher-forced top-3 at only {top3:.3f} of the positions"
        beam = e.generate(B, num_beams=5)
        assert agree >= need, f"{e.dtype}: cached decode vs teacher-forced argmax agreement {agree:.3f}"
        assert ((beam >= 0) & (beam < enc_cfg.vocab_size)).all()


def _padded_history(enc_cfg, B, hist):
    b = history_batch(enc_cfg, 0, B)
    g = torch.Generator().manual_seed(hist)
    ids = b["enc_input_ids"]
    for i in range(B):
        n = int((ids[i] != 0).sum())
        ids[i, n:hist] = torch.randint(1000 if enc_cfg.vocab_size > 2000 else 104, enc_cfg.vocab_size, (hist - n,), generator=g)
    b["enc_att_mask"] = (ids != 0).float()
    return b


@pytest.mark.parametrize("which", ["full", "tiny"])
def test_self_attention_v2_agrees_with_v1(full_cfgs, full_sd, tiny_cfgs, tiny_sd, which):
    """The default bf16 decode self-attention (lean kernel, GSTVD_SELF_V2) against the first kernel inside the same engine: eager
    decode steps, the switches are read per launch.  Greedy and beam token ids must agree (bf16 rounding may flip a near-tie, hence
    >= 90 % / 80 %); reading the history through the beam ancestry table (GSTVD_SELF_ANC, default) must give token ids IDENTICAL
    to gathering the cache after every step (reorder_cache_kernel, visual_dialog_decoder.py:177-181); and the teacher-forced pass
    over the greedy tokens must reproduce them like it does for the first kernel."""
    from gst_visdial_b200 import _lib
    from gst_visdial_b200.engine import Engine
    enc_cfg, dec_cfg = full_cfgs if which == "full" else tiny_cfgs
    sd = full_sd if which == "full" else tiny_sd
    B = 3
    e = Engine(enc_cfg, dec_cfg, dtype="bf16", max_batch=B, max_beams=5, flags=_lib.GSTVD_FLAG_NO_CUDA_GRAPH)
    e.load_state_dict(sd)
    try:
        b = _padded_history(enc_cfg, B, 140)
        o = e.encode(b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"], b["enc_image_mask"])
        e.prefill_cross(B, o["Le"])
        res = {}
        for v, anc in (("0", "0"), ("1", "0"), ("1", "1")):
            os.environ["GSTVD_SELF_V2"], os.environ["GSTVD_SELF_ANC"] = v, anc
            res[v + anc] = (e.generate(B, num_beams=1, top_k=1).cpu(), e.generate(B, num_beams=5).cpu(), e.generate(B, num_beams=2).cpu())
        os.environ["GSTVD_SELF_V2"], os.environ["GSTVD_SELF_ANC"] = "0", "0"
        greedy_agree = (res["00"][0] == res["10"][0]).float().mean().item()
        beam_agree = (res["00"][1] == res["10"][1]).float().mean().item()
        print(f"self-attention v2 vs v1 ({which}): greedy agreement {greedy_agree:.3f}, beam-5 agreement {beam_agree:.3f}")
        assert greedy_agree >= 0.9 and beam_agree >= 0.8
        # ancestry table instead of the per-step cache gather: the same kernel reads the same rows from other slots -> identical ids
        assert torch.equal(res["11"][0], res["10"][0])
        assert torch.equal(res["11"][1], res["10"][1]), (res["11"][1], res["10"][1])
        assert torch.equal(res["11"][2], res["10"][2]), (res["11"][2], res["10"][2])
        # teacher-forced pass (different kernels) over the v2 greedy tokens
        out = res["10"][0]
        dec_in = torch.cat((torch.full((B, 1), 101, dtype=torch.int64), out[:, :-1]), 1).cuda()
        _, lg = e.score(dec_in, None, labels=torch.zeros_like(dec_in), want_logits=True)
        agree = (lg.argmax(-1).cpu() == out).float().mean().item()
        print(f"  teacher-forced argmax reproduces the v2 greedy tokens: {agree:.3f}")
        assert agree >= 0.75
    finally:
        os.environ.pop("GSTVD_SELF_V2", None)
        os.environ.pop("GSTVD_SELF_ANC", None)
        e.close()


# ---- the ten-round loop of generate.py:122-233 (SURVEY.md row a17) ------------------------------------------------------
def test_dialog_loop_matches_reference_loop(tiny_cfgs, tiny_sd):
    """Questioner + teacher alternating rounds with history splices and the perplexity pass, fp32, greedy with 4-gram
    blocking for questions: token ids, final history and abnormal flags identical; ppl within 1e-3 relative."""
    from gst_visdial_b200 import synthetic as S, weights as W
    from gst_visdial_b200.dialog import generate_dialogs
    from oracle import dialog_loop as DL
    enc_cfg, dec_cfg = tiny_cfgs
    sd_q = W.synthetic_state_dict(enc_cfg, dec_cfg, seed=7)
    a_model, _ = _build_model(W.TINY_ENC_CONFIG, W.TINY_DEC_CONFIG, tiny_sd, "fp32", model="enc_dec_a")
    q_model, _ = _build_model(W.TINY_ENC_CONFIG, W.TINY_DEC_CONFIG, sd_q, "fp32", model="enc_dec_q")
    batch = S.synthetic_batch(0, 3, vocab_size=enc_cfg.vocab_size, v_feature_size=enc_cfg.v_feature_size, cap_len=(150, 190))
    kw_a = dict(temperature=1.0, top_k=1, top_p=0.0, ngram_blocking_size=0)
    kw_q = dict(temperature=0.7, top_k=1, top_p=0.0, ngram_blocking_size=4)
    rounds = 3                                     # long captions: the third round overflows 256 tokens for some rows
    rq, ra, rp, rf, rids = DL.generate_dialogs(tiny_sd, enc_cfg, dec_cfg, batch, sd_q=sd_q, num_rounds=rounds, a_kwargs=kw_a, q_kwargs=kw_q)
    res = generate_dialogs(a_model, batch, q_model=q_model, num_rounds=rounds, a_kwargs=kw_a, q_kwargs=kw_q, with_ppl=True)
    assert torch.equal(res.questions.cpu(), rq), f"{res.questions.cpu()} vs {rq}"
    assert torch.equal(res.answers.cpu(), ra)
    assert torch.equal(res.enc_input_ids.cpu(), rids)
    assert torch.equal(res.abnormal.cpu(), rf)
    ok = torch.isfinite(rp)
    assert torch.allclose(res.answer_ppl.cpu()[ok], rp[ok], rtol=1e-3)
    assert rf.any(), "test should exercise the overflow path; lengthen the captions"


def test_dialog_loop_beam_config2_shape(tiny_cfgs, tiny_sd):
    """Config-2 shaped loop (teacher only, synthetic questions, beam 5, no ppl) against the oracle loop, fp32."""
    from gst_visdial_b200 import synthetic as S, weights as W
    from gst_visdial_b200.dialog import generate_dialogs
    from oracle import dialog_loop as DL
    enc_cfg, dec_cfg = tiny_cfgs
    a_model, _ = _build_model(W.TINY_ENC_CONFIG, W.TINY_DEC_CONFIG, tiny_sd, "fp32")
    B, rounds = 3, 3
    batch = S.synthetic_batch(0, B, vocab_size=enc_cfg.vocab_size, v_feature_size=enc_cfg.v_feature_size)
    ques = torch.stack([torch.stack([S.synthetic_utterance(i, r, enc_cfg.vocab_size) for r in range(rounds)]) for i in range(B)])
    kw = dict(temperature=1.0, top_k=1, top_p=0.0, ngram_blocking_size=0, num_beams=5)
    rq, ra, _, rf, rids = DL.generate_dialogs(tiny_sd, enc_cfg, dec_cfg, batch, questions=ques, num_rounds=rounds, a_kwargs=kw, with_ppl=False)
    res = generate_dialogs(a_model, batch, questions=ques, num_rounds=rounds, a_kwargs=kw, with_ppl=False)
    assert torch.equal(res.answers.cpu().masked_fill(res.answers.cpu() == 102, 0), ra)
    assert torch.equal(res.enc_input_ids.cpu(), rids)


def test_history_trimming_is_exact(tiny_cfgs, tiny_sd):
    """Encoder on ceil32(longest history) positions vs all max_seq_len positions: identical ids, ppl, history and flags."""
    from gst_visdial_b200 import synthetic as S, weights as W
    from gst_visdial_b200.dialog import generate_dialogs
    enc_cfg, dec_cfg = tiny_cfgs
    for dtype in ("fp32", "bf16"):
        a_model, _ = _build_model(W.TINY_ENC_CONFIG, W.TINY_DEC_CONFIG, tiny_sd, dtype)
        B, rounds = 4, 4
        batch = S.synthetic_batch(0, B, vocab_size=enc_cfg.vocab_size, v_feature_size=enc_cfg.v_feature_size)
        ques = torch.stack([torch.stack([S.synthetic_utterance(i, r, enc_cfg.vocab_size) for r in range(rounds)]) for i in range(B)])
        kw = dict(temperature=1.0, top_k=1, top_p=0.0, ngram_blocking_size=0, num_beams=3)
        r1 = generate_dialogs(a_model, batch, questions=ques, num_rounds=rounds, a_kwargs=kw, with_ppl=True, trim_history=True)
        r0 = generate_dialogs(a_model, batch, questions=ques, num_rounds=rounds, a_kwargs=kw, with_ppl=True, trim_history=False)
        assert torch.equal(r1.answers, r0.answers) and torch.equal(r1.enc_input_ids, r0.enc_input_ids)
        assert torch.equal(r1.abnormal, r0.abnormal)
        assert torch.equal(r1.answer_ppl.nan_to_num(-1.0), r0.answer_ppl.nan_to_num(-1.0)), dtype


def test_dialog_host_length_hints_are_equivalent(tiny_cfgs, tiny_sd):
    """Device-resident inputs + the optional host copies of the caption / question lengths (`enc_len_host`, `questions_len_host`:
    no device read at the start of a dialog) give exactly what host inputs and plain device inputs give."""
    from gst_visdial_b200 import synthetic as S, weights as W
    from gst_visdial_b200.dialog import generate_dialogs
    enc_cfg, dec_cfg = tiny_cfgs
    a_model, _ = _build_model(W.TINY_ENC_CONFIG, W.TINY_DEC_CONFIG, tiny_sd, "bf16")
    B, rounds = 4, 3
    batch = S.synthetic_batch(0, B, vocab_size=enc_cfg.vocab_size, v_feature_size=enc_cfg.v_feature_size)
    ques = torch.stack([torch.stack([S.synthetic_utterance(i, r, enc_cfg.vocab_size) for r in range(rounds)]) for i in range(B)])
    kw = dict(temperature=1.0, top_k=1, top_p=0.0, ngram_blocking_size=0, num_beams=3)
    ref = generate_dialogs(a_model, batch, questions=ques, num_rounds=rounds, a_kwargs=kw, with_ppl=True)
    dev_batch = {k: v.cuda() for k, v in batch.items()}
    plain = generate_dialogs(a_model, dev_batch, questions=ques.cuda(), num_rounds=rounds, a_kwargs=kw, with_ppl=True)
    hinted = dict(dev_batch, enc_len_host=(batch["enc_input_ids"] != 0).sum(-1), questions_len_host=(ques != 0).sum(-1))
    hint = generate_dialogs(a_model, hinted, questions=ques.cuda(), num_rounds=rounds, a_kwargs=kw, with_ppl=True)
    for r in (plain, hint):
        assert torch.equal(r.answers, ref.answers) and torch.equal(r.enc_input_ids, ref.enc_input_ids) and torch.equal(r.abnormal, ref.abnormal)
        assert torch.equal(r.answer_ppl.nan_to_num(-1.0), ref.answer_ppl.nan_to_num(-1.0))


def test_generate_cli_synthetic(tmp_path):
    """generate.py end to end (questioner + teacher, sampling with 4-gram blocking, ppl) on the tiny configs."""
    import json
    import subprocess
    import sys
    from gst_visdial_b200 import weights as W
    from helpers import ROOT
    cmd = [sys.executable, os.path.join(ROOT, "generate.py"), "-synthetic", "5", "-batch_size", "4", "-num_rounds", "2",
           "-model_enc_config", W.TINY_ENC_CONFIG, "-model_dec_config", W.TINY_DEC_CONFIG, "-save_path", str(tmp_path), "-save_name", "o.json",
           "-compute_dtype", "bf16"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    out = json.load(open(tmp_path / "o.json"))
    assert len(out) == 5 and len(out[0]["dialog"]) == 2 and out[0]["dialog"][0]["answer_ppl"] > 0


def test_generate_cli_feature_shards(tmp_path, tiny_cfgs):
    """generate.py fed from bf16 feature shards + pre-tokenized captions (SURVEY.md row f3), streamed JSONL output (f4)."""
    import json
    import subprocess
    import sys
    from gst_visdial_b200 import synthetic as S, weights as W
    from gst_visdial_b200.io import features as IOF
    from helpers import ROOT
    enc_cfg, _ = tiny_cfgs
    b = S.synthetic_batch(0, 6, vocab_size=enc_cfg.vocab_size, v_feature_size=enc_cfg.v_feature_size)
    ids = [500 + i for i in range(6)]
    IOF.write_shard(str(tmp_path / "s0"), ids[:4], b["enc_image_feat"][:4].numpy(), b["enc_image_loc"][:4].numpy(), b["enc_image_mask"][:4].numpy())
    IOF.write_shard(str(tmp_path / "s1"), ids[4:], b["enc_image_feat"][4:].numpy(), b["enc_image_loc"][4:].numpy(), b["enc_image_mask"][4:].numpy())
    caps = {str(i): [int(t) for t in row[1:] if int(t) not in (0, 102)] for i, row in zip(ids, b["enc_input_ids"].tolist())}
    json.dump(caps, open(tmp_path / "caps.json", "w"))
    cmd = [sys.executable, os.path.join(ROOT, "generate.py"), "-feature_shards", f"{tmp_path / 's0'},{tmp_path / 's1'}", "-caption_ids",
           str(tmp_path / "caps.json"), "-batch_size", "4", "-num_rounds", "2", "-model_enc_config", W.TINY_ENC_CONFIG, "-model_dec_config",
           W.TINY_DEC_CONFIG, "-save_path", str(tmp_path), "-save_name", "o.json", "-compute_dtype", "bf16"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    out = json.load(open(tmp_path / "o.json"))
    assert [d["image_id"] for d in out] == ids and len(out[0]["dialog"]) == 2
    assert out[2]["caption"] == " ".join(str(t) for t in [101] + caps["502"] + [102])
    assert sum(1 for _ in open(tmp_path / "o.json.jsonl")) == 6


def test_generative_ranking_shares_encoder(tiny_fp32, tiny_cfgs, tiny_sd):
    """f1 (evaluate_gen.py:62-107): O options per image scored against one encoder pass == scoring every option separately."""
    from gst_visdial_b200.ranking import score_options
    model, _ = tiny_fp32
    enc_cfg, dec_cfg = tiny_cfgs
    B, O, L = 2, 4, 12
    b = history_batch(enc_cfg, 0, B)
    g = torch.Generator().manual_seed(3)
    opts = torch.zeros(B, O, L, dtype=torch.int64)
    for i in range(B):
        for o in range(O):
            n = int(torch.randint(3, L - 1, (1,), generator=g))
            opts[i, o, 0] = 101
            opts[i, o, 1:n] = torch.randint(104, enc_cfg.vocab_size, (n - 1,), generator=g)
            opts[i, o, n] = 102
    scores = score_options(model, b, opts).cpu()
    with torch.no_grad():
        t, v = R.encoder(tiny_sd, enc_cfg, b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"], b["enc_image_mask"])
        eh, em = R.vlfusion(tiny_sd, t, v, b["enc_att_mask"], b["enc_image_mask"])
        ids = opts.reshape(B * O, L)
        labels = torch.zeros_like(ids); labels[:, :-1] = ids[:, 1:]
        logits = R.lm_logits(tiny_sd, R.decoder_hidden(tiny_sd, dec_cfg, ids, (ids != 0).float(), eh.repeat_interleave(O, 0), em.repeat_interleave(O, 0)))
        lp = torch.log_softmax(logits, -1).gather(-1, labels.unsqueeze(-1)).squeeze(-1) * (labels != 0).float()
        ref = lp.sum(-1).reshape(B, O)
    assert max_abs(scores, ref) < 2e-3
    assert torch.equal(scores.argsort(-1), ref.argsort(-1))


def test_answer_perplexity_config4(tiny_fp32, tiny_cfgs, tiny_sd):
    """Config 4 (-select_data scoring): teacher-forced ppl of given answers == generate.py:183-209 restated."""
    from gst_visdial_b200.ranking import answer_perplexity, select_mask
    model, _ = tiny_fp32
    enc_cfg, dec_cfg = tiny_cfgs
    B = 3
    b = history_batch(enc_cfg, 0, B)
    g = torch.Generator().manual_seed(11)
    ans = torch.zeros(B, 18, dtype=torch.int64)
    for i, n in enumerate((18, 7, 1)):                 # full length without [SEP], [SEP]-terminated, lone [SEP] (NaN ppl)
        ans[i, :n] = torch.randint(104, enc_cfg.vocab_size, (n,), generator=g)
    ans[1, 6] = 102
    ans[2, 0] = 102
    ppl = answer_perplexity(model, b, ans).cpu()
    with torch.no_grad():
        _, _, ref = R.score_answers(tiny_sd, enc_cfg, dec_cfg, b, ans)
    ok = torch.isfinite(ref)
    assert torch.equal(torch.isfinite(ppl), ok) and ok.tolist() == [True, True, False]
    assert torch.allclose(ppl[ok], ref[ok], rtol=1e-3)
    thr = float(ref[ok].mean())
    assert torch.equal(select_mask(ppl, thr), ~(ref >= thr))


def test_nsp_rank_config5(tiny_cfgs, tiny_sd):
    """Config 5 (evaluate_disc.py:79-83): softmax(nsp)[:, 0] per candidate row, and the ranking it induces."""
    from gst_visdial_b200 import weights as W
    from gst_visdial_b200.models.visual_dialog_encoder import VisualDialogEncoder
    from gst_visdial_b200.ranking import nsp_rank
    enc_cfg, _ = tiny_cfgs
    params = _params(W.TINY_ENC_CONFIG, W.TINY_DEC_CONFIG, "fp32", model="enc_only_a", mode="vd_eval_val")
    enc = VisualDialogEncoder(params)
    enc.load_state_dict({k[len("encoder."):]: v for k, v in tiny_sd.items() if k.startswith("encoder.")})
    enc.to("cuda:0").eval()
    n_opt = 6
    b = history_batch(enc_cfg, 0, 1)
    g = torch.Generator().manual_seed(5)
    tokens = b["enc_input_ids"].repeat(n_opt, 1)
    seg = b["enc_segments"].repeat(n_opt, 1)
    n0 = int((tokens[0] != 0).sum())
    for o in range(n_opt):                              # each candidate appended to the text stream (dataloader_visdial_disc.py:320-323)
        n = 3 + o
        tokens[o, n0:n0 + n] = torch.randint(104, enc_cfg.vocab_size, (n,), generator=g)
        tokens[o, n0 + n] = 102
        seg[o, n0:n0 + n + 1] = 1
    item = dict(tokens=tokens, segments=seg, mask=(tokens != 0).float(), image_feat=b["enc_image_feat"].repeat(n_opt, 1, 1),
                image_loc=b["enc_image_loc"].repeat(n_opt, 1, 1), image_mask=b["enc_image_mask"].repeat(n_opt, 1))
    p = nsp_rank(enc, item).cpu()
    with torch.no_grad():
        t, v = R.encoder(tiny_sd, enc_cfg, tokens, item["image_feat"], item["image_loc"], seg, item["mask"], item["image_mask"])
        ref = torch.softmax(R.nsp_scores(tiny_sd, t, v), 1)[:, 0]
    assert max_abs(p, ref) < 1e-3
    assert torch.equal(p.argsort(descending=True), ref.argsort(descending=True))


# ---- edges and error behaviour ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,K", [(1, 8), (4, 1), (2, 2)])
def test_tiny_fp32_beam_widths_match_oracle(tiny_cfgs, tiny_sd, B, K):
    """Smallest batch with the widest beam the kernels support (8); beam 1 (served by the greedy path: same tokens); beam 2."""
    from gst_visdial_b200.engine import Engine
    enc_cfg, dec_cfg = tiny_cfgs
    e = Engine(enc_cfg, dec_cfg, dtype="fp32", max_batch=B, max_beams=K)
    e.load_state_dict(tiny_sd)
    b = history_batch(enc_cfg, 10, B)
    with torch.no_grad():
        ref_seq, ref_sc = OB.beam_search(tiny_sd, enc_cfg, dec_cfg, b, num_beams=K)
    o = e.encode(b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"], b["enc_image_mask"])
    e.prefill_cross(B, o["Le"])
    seq, sc = e.generate(B, num_beams=K, want_scores=True)
    assert torch.equal(seq.cpu(), ref_seq)
    if K > 1:                                             # num_beams = 1 takes the greedy path, which keeps no hypothesis scores
        assert torch.allclose(sc.cpu().double(), ref_sc, atol=1e-4)
    e.close()


def test_capacity_and_state_errors_are_reported(tiny_cfgs, tiny_sd):
    """The C ABI reports misuse through status codes + gstvd_last_error (raised as GstvdError), it never writes out of bounds."""
    from gst_visdial_b200._lib import GstvdError
    from gst_visdial_b200.engine import Engine
    enc_cfg, dec_cfg = tiny_cfgs
    e = Engine(enc_cfg, dec_cfg, dtype="bf16", max_batch=2, max_beams=2)
    b = history_batch(enc_cfg, 0, 3)
    args = (b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"], b["enc_image_mask"])
    with pytest.raises(GstvdError):                       # weights not loaded yet
        e.encode(*[a[:2] for a in args])
    e.load_state_dict(tiny_sd)
    with pytest.raises(GstvdError, match="capacity"):     # 3 images into a context sized for 2
        e.encode(*args)
    with pytest.raises(GstvdError):                       # nothing prefilled yet
        e.generate(2, num_beams=2)
    o = e.encode(*[a[:2] for a in args])
    e.prefill_cross(2, o["Le"])
    with pytest.raises(GstvdError, match="num_beams"):    # wider than the context was built for
        e.generate(2, num_beams=5)
    with pytest.raises(GstvdError):                       # prefilled for 2 images, asked for 1
        e.generate(1, num_beams=2)
    with pytest.raises(GstvdError):                       # top_k outside 0..16
        e.generate(2, num_beams=1, top_k=17, top_p=0.9, temperature=1.0)
    ids0 = e.generate(2, num_beams=1, top_k=0, top_p=0.9, temperature=1.0, seed=3)   # top_k = 0: pure nucleus over the vocabulary
    assert ids0.shape == (2, 18) and int(ids0.min()) >= 0 and int(ids0.max()) < enc_cfg.vocab_size
    assert torch.equal(ids0, e.generate(2, num_beams=1, top_k=0, top_p=0.9, temperature=1.0, seed=3))
    ids = e.generate(2, num_beams=2)                      # and the context still works afterwards
    assert ids.shape == (2, 18)
    e.close()


def test_score_max_length_and_single_token(tiny_fp32, tiny_cfgs, tiny_sd):
    """Teacher-forced pass at the longest decoder input the context accepts (max_utt_len = 25) and at length 1."""
    model, _ = tiny_fp32
    enc_cfg, dec_cfg = tiny_cfgs
    B = 2
    b = history_batch(enc_cfg, 0, B)
    eng = model.module._engine(torch.device("cuda:0"))
    o = eng.encode(b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"], b["enc_image_mask"])
    eng.prefill_cross(B, o["Le"])
    with torch.no_grad():
        t, v = R.encoder(tiny_sd, enc_cfg, b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"], b["enc_image_mask"])
        eh, em = R.vlfusion(tiny_sd, t, v, b["enc_att_mask"], b["enc_image_mask"])
    g = torch.Generator().manual_seed(9)
    for L in (25, 1):
        ids = torch.randint(104, enc_cfg.vocab_size, (B, L), generator=g)
        ids[:, 0] = 101
        _, lg = eng.score(ids.cuda(), None, labels=torch.zeros(B, L, dtype=torch.int64).cuda(), want_logits=True)
        with torch.no_grad():
            ref = R.lm_logits(tiny_sd, R.decoder_hidden(tiny_sd, dec_cfg, ids, torch.ones(B, L), eh, em))
        assert max_abs(lg.cpu(), ref) < FP32_LOGIT_TOL


def test_evaluate_gen_cli_synthetic(tmp_path):
    """evaluate_gen.py end to end on the tiny configs: ranks json in the reference's layout + sparse metrics."""
    import json
    import subprocess
    import sys
    from gst_visdial_b200 import weights as W
    from helpers import ROOT
    cmd = [sys.executable, os.path.join(ROOT, "evaluate_gen.py"), "-synthetic", "3", "-num_options", "7", "-num_rounds", "2", "-batch_size", "14",
           "-model_enc_config", W.TINY_ENC_CONFIG, "-model_dec_config", W.TINY_DEC_CONFIG, "-save_path", str(tmp_path), "-save_name", "r.json",
           "-compute_dtype", "fp32"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    out = json.load(open(tmp_path / "r.json"))
    assert len(out) == 6 and sorted(out[0]["ranks"]) == list(range(1, 8)) and {d["round_id"] for d in out} == {1, 2}
    m = json.loads(r.stdout.strip().splitlines()[-1])
    assert 0.0 <= m["mrr"] <= 1.0 and 1.0 <= m["mean"] <= 7.0


def test_bench_dump_outputs(tmp_path):
    """bench.py --dump-outputs writes the last timed step's results as .npy files (select_data: the fp32 perplexities); the JSON line
    reports the requested number of timed steps."""
    import json
    import subprocess
    import sys
    from helpers import ROOT
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "select_data", "--batch", "8", "--steps", "3", "--warmup", "1",
           "--no-cpu-baseline", "--dump-outputs", str(tmp_path / "out")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout + r.stderr
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 3 and line["config"]["output_check"]["deterministic"] is True
    assert sorted(os.listdir(tmp_path / "out")) == ["answer_ppl.npy"]
    ppl = np.load(tmp_path / "out" / "answer_ppl.npy")
    assert ppl.dtype == np.float32 and ppl.shape == (8,) and np.isfinite(ppl).all() and (ppl > 1).all()


def test_pair_gemm_encoder_prefill_match_single(full_cfgs, full_sd):
    """Whole encoder, cross-K/V prefill (head-major TMA-store epilogue) and the decode that reads the cache with the CTA-pair GEMM
    forced on every eligible problem against the single-CTA kernel: outputs within bf16 noise, token ids identical."""
    from gst_visdial_b200.engine import Engine
    enc_cfg, dec_cfg = full_cfgs
    B = 8
    e = Engine(enc_cfg, dec_cfg, dtype="bf16", max_batch=B, max_beams=5)
    e.load_state_dict(full_sd)
    try:
        b = history_batch(enc_cfg, 0, B)
        outs = []
        for flag in ("0", "256"):
            os.environ["GSTVD_GEMM_2CTA"] = flag
            try:
                o = e.encode(b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"],
                             b["enc_image_mask"], want_t=True, want_v=True, want_fused=True)
                e.prefill_cross(B, o["Le"])
            finally:
                os.environ.pop("GSTVD_GEMM_2CTA", None)
            outs.append((o["seq_t"].cpu(), o["seq_v"].cpu(), o["fused"].cpu(), e.generate(B, num_beams=1, top_k=1).cpu(),
                         e.generate(B, num_beams=5).cpu()))
        for x0, x1 in zip(outs[0][:3], outs[1][:3]):
            assert torch.isfinite(x1).all() and rel_rms(x1, x0) < 1e-3, rel_rms(x1, x0)
        assert torch.equal(outs[0][3], outs[1][3]) and torch.equal(outs[0][4], outs[1][4])
    finally:
        e.close()
