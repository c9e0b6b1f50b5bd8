"""Ten-round synthetic dialog generation: the loop of the reference's generate.py:122-233 without its host syncs.

Per round: question (questioner model, or a caller-supplied utterance) -> splice into the history ->
answer (teacher model) -> optional perplexity pass over the answer (generate.py:183-209) -> splice the answer with
segment 1.  History state stays on the device; the splices run in the engine's integer kernels (gstvd_splice), so
nothing in a round waits for the host.

Reference quirks kept (SURVEY.md section 8a): the answer reaches the history WITHOUT its [SEP] (the perplexity pass
replaces [SEP] by [PAD] in place before the splice, single-device behaviour); overflow past max_seq_len writes a
lone [SEP] and marks the dialog abnormal; ppl = exp(sum CE / count(ids != 0)) with the first answer token unscored.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional

import torch


@dataclass
class DialogResult:
    questions: torch.Tensor      # int64 [B, rounds, 18]
    answers: torch.Tensor        # int64 [B, rounds, 18]  ([SEP] already replaced by [PAD] when ppl was computed)
    answer_ppl: Optional[torch.Tensor]   # fp32 [B, rounds] or None
    abnormal: torch.Tensor       # int32 [B] (1 = history overflowed, dropped from the output like generate.py:236-237)
    enc_input_ids: torch.Tensor  # final history [B, max_seq_len]


def _unwrap(model):
    return model.module if hasattr(model, "module") else model


def _model_call(model, st, dec_input_ids, **kw):
    return model(
        enc_image_features=st["feat"], enc_image_spatials=st["loc"], enc_image_mask=st["imask"], enc_image_target=None,
        enc_image_label=None, enc_next_sentence_labels=None, enc_input_ids=st["ids"], enc_segments=st["seg"], enc_sep_indices=None,
        enc_mlm_labels=None, enc_attention_mask=st["mask"], dec_input_ids=dec_input_ids,
        dec_attention_mask=(dec_input_ids != 0).float(), **kw)


def _answer_ppl(a_model, st, ans, mode):
    """Perplexity pass of generate.py:183-209 over ``ans`` [B, 18] against the resident cross-K/V; replaces [SEP] by [PAD] in place."""
    am = _unwrap(a_model)
    am.params["mode"] = "train"                              # the reference's mode-flip trick (generate.py:185,211)
    try:
        loss, _ = _model_call(a_model, st, ans, loss_reduction=False, reuse_encoder=True, want_logits=False)
    finally:
        am.params["mode"] = mode
    ans_len = (ans != 0).sum(-1)                             # counted after the in-place [SEP] -> [PAD]
    return torch.exp(loss.reshape(ans.shape[0], -1).sum(-1) / ans_len)


def _best_candidate(a_model, st, cands, mode):
    """cands [B, N, 18]: every candidate through the perplexity pass, then per image the one with the lowest perplexity (a stable
    ascending sort puts NaN last and keeps the lowest candidate index among ties).  Returns (answers [B, 18], perplexities [B])."""
    B, N, L = cands.shape
    rows = [cands[:, n].contiguous() for n in range(N)]
    ppl = torch.stack([_answer_ppl(a_model, st, r, mode) for r in rows], 1)
    best = torch.sort(ppl, dim=1, stable=True).indices[:, :1]
    ans = torch.stack(rows, 1).gather(1, best[:, :, None].expand(B, 1, L)).squeeze(1)
    return ans, ppl.gather(1, best).squeeze(1)


def generate_dialogs(a_model, batch, q_model=None, questions=None, num_rounds=10, a_kwargs=None, q_kwargs=None,
                     with_ppl=True, device=None, trim_history=True, max_new_tokens=18, seed=None, row_offset=0,
                     answer_candidates=1) -> DialogResult:
    """``batch`` uses the reference dataloader's keys (generate.py:95-111).  Either ``q_model`` or ``questions``
    (int64 [B, num_rounds, 18], zero padded, each ending in [SEP]) must be given.  ``a_kwargs`` / ``q_kwargs`` are the
    decoding kwargs of EncoderDecoderModel.forward; defaults are generate.py:138-141 / :177-180.

    Optional keys ``enc_len_host`` (int64 [B], non-pad tokens of ``enc_input_ids``) and ``questions_len_host`` ([B, rounds]) are
    HOST copies of the lengths the history bound starts from; with device-resident inputs they avoid the one device read (a stream
    drain) at the start of a dialog.  They must be upper bounds of the true lengths.

    ``trim_history``: the encoder runs on ceil32(longest history) text positions instead of all ``max_seq_len`` (see
    ``enc_valid_len`` in EncoderDecoderModel.forward).  The bound is kept on the HOST - caption lengths are read once at the
    start, every round adds the question length (or ``max_new_tokens`` for a generated question) and ``max_new_tokens`` for
    the answer - so no round waits for the device.  Token ids, perplexities and flags are identical with or without it.

    ``answer_candidates`` > 1 (needs ``with_ppl``): per round the teacher draws that many answers in one call (samples, or the best of
    its ``num_beams`` beams), and the one with the lowest perplexity is spliced and reported."""
    a_kwargs = dict(a_kwargs or dict(temperature=0.7, top_k=7, top_p=0.0, ngram_blocking_size=0))
    q_kwargs = dict(q_kwargs or dict(temperature=0.7, top_k=7, top_p=0.0, ngram_blocking_size=4))
    am = _unwrap(a_model)
    dev = torch.device(device) if device is not None else next(am.parameters()).device
    eng = am._engine(dev)
    nb = dict(device=dev, non_blocking=True)
    st = {
        # features travel in their own dtype (bf16 shards: 152 KB / image) and are widened on the device
        "feat": batch["enc_image_feat"].to(**nb).to(torch.float32), "loc": batch["enc_image_loc"].to(dtype=torch.float32, **nb),
        "imask": batch["enc_image_mask"].to(dtype=torch.float32, **nb),
        "ids": batch["enc_input_ids"].to(dtype=torch.int64, **nb).clone().contiguous(),
        "seg": batch["enc_segments"].to(dtype=torch.int64, **nb).clone().contiguous(),
    }
    B = st["ids"].shape[0]
    st["mask"] = (st["ids"] != 0).float()
    enc_len = (st["ids"] != 0).sum(-1).to(torch.int32)
    abnormal = torch.zeros(B, dtype=torch.int32, device=dev)
    dec_start = batch["dec_input_ids"].to(dtype=torch.int64, **nb)
    q_host = None                                               # [B, rounds] question lengths, read before the copy to the device
    if questions is not None:
        if trim_history and q_model is None:
            q_host = batch.get("questions_len_host")            # optional: lengths the caller already holds on the host
            if q_host is None:
                q_host = (questions != 0).sum(-1).cpu().to(torch.int64)
        questions = questions.to(dtype=torch.int64, **nb)
    elif q_model is None:
        raise ValueError("generate_dialogs needs q_model or questions")
    n_cand = int(answer_candidates)
    if n_cand < 1 or (n_cand > 1 and not with_ppl):
        raise ValueError("answer_candidates must be >= 1, and more than one candidate is ranked by perplexity (with_ppl=True)")
    ques_all, ans_all, ppl_all = [], [], []
    mode = am.params["mode"]
    Lmax = st["ids"].shape[1]
    ub = None                                                   # host-side per-row upper bound of the history length
    if trim_history:
        ub = batch.get("enc_len_host")                          # optional host copy of the caption lengths (int64 [B])
        if ub is None:
            ub = (batch["enc_input_ids"] != 0).sum(-1).cpu().to(torch.int64)  # one read at the start (free for host inputs)
        ub = ub.to(torch.int64).clone()

    def bound():
        return int(ub.max().clamp(max=Lmax)) if ub is not None else None

    from .models.visual_dialog_model import derive_seed
    base_seed = am.params.get("seed", 0) if seed is None else seed
    a_user, q_user = a_kwargs, q_kwargs
    for rnd in range(num_rounds):
        a_kwargs = a_user if "seed" in a_user else dict(a_user, seed=derive_seed(base_seed, "a", rnd), row_offset=row_offset)
        if q_model is None:
            ques = questions[:, rnd].contiguous()
        else:
            qk = q_user if "seed" in q_user else dict(q_user, seed=derive_seed(base_seed, "q", rnd), row_offset=row_offset)
            ques = _model_call(q_model, st, dec_start, enc_valid_len=bound(), **qk)
        eng.splice(st["ids"], st["seg"], st["mask"], enc_len, ques, segment_value=-1, strip_sep=False, abnormal=abnormal)
        if ub is not None:
            ub = ub + (q_host[:, rnd] if q_host is not None else max_new_tokens)
        if n_cand > 1:
            cands = _model_call(a_model, st, dec_start, enc_valid_len=bound(), num_return_sequences=n_cand, **a_kwargs)
        else:
            ans = _model_call(a_model, st, dec_start, enc_valid_len=bound(), **a_kwargs)
        if ub is not None:
            ub = ub + max_new_tokens
        if n_cand > 1:
            ans, ppl = _best_candidate(a_model, st, cands.reshape(B, n_cand, -1), mode)
            ppl_all.append(ppl)
        elif with_ppl:
            ppl_all.append(_answer_ppl(a_model, st, ans, mode))
        eng.splice(st["ids"], st["seg"], st["mask"], enc_len, ans, segment_value=1, strip_sep=True, abnormal=abnormal)
        ques_all.append(ques)
        ans_all.append(ans)
    return DialogResult(torch.stack(ques_all, 1), torch.stack(ans_all, 1), torch.stack(ppl_all, 1) if with_ppl else None,
                        abnormal, st["ids"])
