"""TEST INFRASTRUCTURE ONLY - generates tests/golden/*.npz by running the REFERENCE'S OWN classes.

Run in the development container only (needs /root/reference):  ``python -m oracle.gen_golden``

For each case it
  1. builds seeded weights (gst_visdial_b200.weights.synthetic_state_dict) and checks the key/shape spec against the
     state_dict registered by the reference constructors (strict load),
  2. runs the reference ``EncoderDecoderModel`` / ``VisualDialogEncoder`` (under oracle/ref_shim.py) on seeded
     synthetic inputs: greedy decode through the reference sampler (top_k=1), the teacher-forced perplexity pass of
     generate.py:183-209, greedy with 4-gram blocking, and the enc_only NSP scores,
  3. asserts that oracle/restatement.py reproduces the reference outputs (this is what pins the oracle),
  4. writes the reference outputs as small fixtures.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from gst_visdial_b200 import synthetic as S  # noqa: E402
from gst_visdial_b200 import weights as W  # noqa: E402
from oracle import ref_shim  # noqa: E402
from oracle import restatement as R  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
PART_BYTES = 960_000        # uncompressed bytes per golden file: keeps every committed file under 1 MB


def save_golden(tag: str, out: dict) -> list:
    """Writes ``out`` as tests/golden/<tag>.npz and, for the arrays that do not fit, <tag>.part2.npz, <tag>.part3.npz, ...
    (tests/helpers.py:load_golden merges them).  Returns the paths written."""
    parts, size = [{}], 0
    for k, v in out.items():
        if parts[-1] and size + v.nbytes > PART_BYTES:
            parts.append({})
            size = 0
        parts[-1][k] = v
        size += v.nbytes
    os.makedirs(GOLDEN, exist_ok=True)
    paths = [os.path.join(GOLDEN, f"{tag}.npz" if i == 0 else f"{tag}.part{i + 1}.npz") for i in range(len(parts))]
    for path, part in zip(paths, parts):
        np.savez_compressed(path, **part)
    return paths


def history_batch(enc_cfg, start, count, rounds=2):
    """Synthetic batch whose text already holds ``rounds`` (question, answer) pairs, with a repeated question
    4-gram so that n-gram blocking has something to ban."""
    b = S.synthetic_batch(start, count, vocab_size=enc_cfg.vocab_size, v_feature_size=enc_cfg.v_feature_size)
    ids, seg = b["enc_input_ids"], b["enc_segments"]
    enc_len = (ids != 0).sum(-1)
    abnormal = set()
    for r in range(rounds):
        q = torch.stack([S.synthetic_utterance(start + i, 2 * r, enc_cfg.vocab_size) for i in range(count)])
        enc_len += R.splice(ids, seg, enc_len, q, None, abnormal)
        a = torch.stack([S.synthetic_utterance(start + i, 2 * r + 1, enc_cfg.vocab_size) for i in range(count)])
        a = a.masked_fill(a == R.EOS, 0)  # answers are spliced without [SEP] (single-device reference behaviour)
        enc_len += R.splice(ids, seg, enc_len, a, 1, abnormal)
    b["enc_att_mask"] = (ids != 0).float()
    return b


def call_ref(model, b, dec_ids=None, **kw):
    dec = b["dec_input_ids"].clone() if dec_ids is None else dec_ids
    return model(enc_image_features=b["enc_image_feat"], enc_image_spatials=b["enc_image_loc"],
                 enc_image_mask=b["enc_image_mask"], enc_input_ids=b["enc_input_ids"].clone(),
                 enc_segments=b["enc_segments"].clone(), enc_attention_mask=b["enc_att_mask"].clone(),
                 dec_input_ids=dec, dec_attention_mask=(dec != 0).float(), **kw)


def run_case(tag, enc_path, dec_path, batch_size, full_dump):
    enc_cfg, dec_cfg = W.load_json_config(enc_path), W.load_json_config(dec_path)
    sd = W.synthetic_state_dict(enc_cfg, dec_cfg, seed=0)
    model, params = ref_shim.build_reference_model(enc_path, dec_path, model="enc_dec_a", mode="cc12m_gen")
    spec = W.model_spec(enc_cfg, dec_cfg)
    ref_sd = model.state_dict()
    assert set(ref_sd.keys()) == set(spec.keys()), "key layout differs from the reference"
    for k, shp in spec.items():
        assert tuple(ref_sd[k].shape) == tuple(shp), k
    model.load_state_dict(sd, strict=True)
    out = {}
    with torch.no_grad():
        b = history_batch(enc_cfg, 0, batch_size)
        # encoder + fusion through the reference modules
        _, _, _, _, _, seq_t, seq_v = model.encoder(b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"],
                                                    token_type_ids=b["enc_segments"], attention_mask=b["enc_att_mask"],
                                                    image_attention_mask=b["enc_image_mask"])
        fused, fmask = model.vlfusion(seq_t, seq_v, b["enc_att_mask"], b["enc_image_mask"])
        r_t, r_v = R.encoder(sd, enc_cfg, b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"],
                             b["enc_segments"], b["enc_att_mask"], b["enc_image_mask"])
        r_fused, r_fmask = R.vlfusion(sd, r_t, r_v, b["enc_att_mask"], b["enc_image_mask"])
        for name, a, c in (("seq_t", seq_t, r_t), ("seq_v", seq_v, r_v), ("fused", fused, r_fused)):
            err = (a - c).abs().max().item()
            print(f"[{tag}] restatement vs reference {name}: max abs diff {err:.3e}")
            assert err < 2e-4, name
        assert torch.equal(fmask, r_fmask)

        # greedy decode through the reference's own sampler (top_k=1), no blocking
        seq = call_ref(model, b, temperature=1.0, top_k=1, top_p=0.0, ngram_blocking_size=0)
        r_seq, r_logits = R.generate_greedy_or_sample(sd, enc_cfg, dec_cfg, b, 1.0, 1, 0.0, 0, return_logits=True)
        print(f"[{tag}] greedy ids equal: {torch.equal(seq, r_seq)}")
        assert torch.equal(seq, r_seq)
        # greedy with 4-gram blocking against the question history
        seq_ng = call_ref(model, b, temperature=0.7, top_k=1, top_p=0.0, ngram_blocking_size=4)
        r_seq_ng = R.generate_greedy_or_sample(sd, enc_cfg, dec_cfg, b, 0.7, 1, 0.0, 4)
        assert torch.equal(seq_ng, r_seq_ng)
        # reference logits along the greedy path: teacher-force [CLS]+seq[:-1] through the reference decoder
        dec_in = torch.cat((b["dec_input_ids"], seq[:, :-1]), 1)
        params["mode"] = "train"
        _, ref_logits = call_ref(model, b, dec_ids=dec_in.clone(), loss_reduction=False)
        err = (ref_logits - r_logits).abs().max().item()
        print(f"[{tag}] greedy-path logits: max abs diff {err:.3e}")
        assert err < 2e-3
        # perplexity pass exactly as generate.py:185-209
        ans = seq.clone()
        loss, logits = call_ref(model, b, dec_ids=ans, loss_reduction=False)   # mutates ans in place (EOS->PAD)
        params["mode"] = "cc12m_gen"
        ans_len = (ans != 0).sum(-1)
        loss = loss.reshape(batch_size, -1)
        ppl = torch.exp(loss.sum(-1) / ans_len)
        r_loss, r_sl, r_ppl = R.score_answers(sd, enc_cfg, dec_cfg, b, seq)
        assert (loss - r_loss).abs().max().item() < 2e-3 and (logits - r_sl).abs().max().item() < 2e-3
        print(f"[{tag}] ppl ref {ppl.tolist()} restatement {r_ppl.tolist()}")

        # enc_only NSP scores through the reference encoder wrapper
        enc_only, _ = ref_shim.build_reference_model(enc_path, dec_path, model="enc_only_a", mode="vd_eval_val")
        enc_only.load_state_dict({k[len("encoder."):]: v for k, v in sd.items() if k.startswith("encoder.")}, strict=True)
        _, _, _, nsp, _, _, _ = enc_only(b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"],
                                         token_type_ids=b["enc_segments"], attention_mask=b["enc_att_mask"],
                                         image_attention_mask=b["enc_image_mask"])
        r_nsp = R.nsp_scores(sd, r_t, r_v)
        assert (nsp - r_nsp).abs().max().item() < 2e-4
        print(f"[{tag}] nsp ref {nsp.tolist()}")

    out["greedy_ids"] = seq.numpy()
    out["greedy_ng4_ids"] = seq_ng.numpy()
    out["score_loss"] = loss.numpy()
    out["score_ppl"] = ppl.numpy()
    out["nsp"] = nsp.numpy()
    out["enc_input_ids"] = b["enc_input_ids"].numpy().astype(np.int32)
    out["enc_segments"] = b["enc_segments"].numpy().astype(np.int8)
    if full_dump:
        out["seq_t"] = seq_t.numpy(); out["seq_v"] = seq_v.numpy(); out["fused"] = fused.numpy()
        out["greedy_logits"] = ref_logits.numpy()
        out["score_logits"] = logits.numpy()
    else:
        # slices + statistics: enough to catch any layout / arithmetic error without committing megabytes
        out["seq_t_slice"] = seq_t[:, :48, :32].numpy(); out["seq_v_slice"] = seq_v[:, :, :32].numpy()
        out["fused_slice"] = fused[:, :, :24].numpy()
        out["seq_t_rowsum"] = seq_t.sum(-1).numpy(); out["seq_v_rowsum"] = seq_v.sum(-1).numpy()
        out["fused_rowsum"] = fused.sum(-1).numpy()
        out["greedy_logits_slice"] = ref_logits[:, :, :256].numpy()
        top = ref_logits.topk(8, dim=-1)
        out["greedy_logits_top_val"] = top.values.numpy(); out["greedy_logits_top_idx"] = top.indices.numpy().astype(np.int32)
        out["greedy_logits_lse"] = torch.logsumexp(ref_logits, -1).numpy()
    for path in save_golden(tag, out):
        print(f"[{tag}] wrote {path} ({os.path.getsize(path) / 1e6:.2f} MB)")


def main():
    torch.manual_seed(0)
    torch.set_num_threads(os.cpu_count() or 1)
    run_case("tiny_b3", W.TINY_ENC_CONFIG, W.TINY_DEC_CONFIG, 3, full_dump=True)
    if "--tiny-only" not in sys.argv:
        run_case("full_b1", W.DEFAULT_ENC_CONFIG, W.DEFAULT_DEC_CONFIG, 1, full_dump=False)


if __name__ == "__main__":
    main()
