"""Drop-in ``EncoderDecoderModel`` / ``VLFusion`` (reference: models/visual_dialog_model.py:8-135) on the CUDA engine."""
from __future__ import annotations

import torch
from torch import nn

from .. import weights as W
from ._tree import build_tree
from .visual_dialog_decoder import Seq2SeqLMOutput
from .visual_dialog_encoder import _EngineOwner


def _splitmix64(x: int) -> int:
    x = (x + 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF
    x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & 0xFFFFFFFFFFFFFFFF
    x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & 0xFFFFFFFFFFFFFFFF
    return x ^ (x >> 31)


def derive_seed(base, role, index) -> int:
    """64-bit sampling seed from the run seed, the model role ('enc_dec_q' / 'enc_dec_a' ...) and a counter (call or round)."""
    tag = 0xCBF29CE484222325
    for ch in str(role).encode():                      # FNV-1a over the whole role string
        tag = ((tag ^ ch) * 0x100000001B3) & 0xFFFFFFFFFFFFFFFF
    return _splitmix64(_splitmix64(int(base) & 0xFFFFFFFFFFFFFFFF) ^ _splitmix64(tag) ^ ((int(index) + 1) * 0x632BE59BD9B4E019 & 0xFFFFFFFFFFFFFFFF))


def candidate_seed(seed, n) -> int:
    """Sampling seed of candidate ``n`` of an image in a ``num_return_sequences`` call: candidate n draws what a single-sample call
    with this seed draws (mirror of candidate_seed in csrc/select.cu).  Candidate 0 keeps ``seed``."""
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    if int(n) == 0:
        return seed
    return _splitmix64(seed ^ _splitmix64((int(n) * 0xD1B54A32D192ED03) & 0xFFFFFFFFFFFFFFFF))


class VLFusion(nn.Module):
    """Parameters of models/visual_dialog_model.py:123-129; the projection itself runs inside the engine."""

    def __init__(self, config):
        super().__init__()
        self.config = config
        tree = build_tree(W.fusion_spec(config, prefix="vlfusion."), "vlfusion.")
        self.fc_l = tree._modules["fc_l"]
        self.fc_v = tree._modules["fc_v"]


class EncoderDecoderModel(_EngineOwner, nn.Module):
    """Convenience wrapper module, wrapping Encoder and Decoder modules (same contract as the reference).

    Extra keyword arguments (all default to the reference behaviour):
      num_beams=1        >1 switches the token selection to beam search (contract: oracle/beam.py)
      num_return_sequences=1  N sequences per image, image-major [B*N, 18]: the N best beams (oracle/beam_nbest.py), or N sampled
                         candidates, candidate n drawing like a single-sample call with seed candidate_seed(seed, n)
      num_beam_groups=1, diversity_penalty=0.0   diverse beam search (HF names): the num_beams beams in num_beam_groups groups with a
                         Hamming penalty between groups (contract: oracle/beam_groups.py); groups need num_beams > 1
      do_sample=False    with num_beams > 1: beam sampling (HF beam_sample; contract: oracle/beam_sample.py) with temperature / top_k /
                         top_p; num_return_sequences = N runs N independent searches per image, search n seeded candidate_seed(seed, n).
                         Beam groups cannot be combined with it (HF rejects that too).  With num_beams = 1 the sampler runs either way
      repetition_penalty=1.0, no_repeat_ngram_size=0, min_length=0   HF's logits processors (HF names; 1 / 0 / 0 = off) on each row's
                         own decoder input, dec_input_ids included; min_length counts the decoder input, not new tokens (contract:
                         oracle/processors.py and gstvd_generate in include/gstvd.h)
      length_penalty=1.0, early_stopping=False   HF's beam hypothesis scoring (HF names and defaults): score = sum / len ** length_penalty,
                         is_done as soon as num_beams hypotheses are finished with early_stopping; beam modes only (oracle/decode_args.py)
      bad_words_ids=None   HF-style list of id lists the output never completes, every mode (oracle/decode_args.py)
      seed=None          sampling seed (a per-call counter when None)
      enc_valid_len=None   upper bound (python int) on the number of leading history positions that hold a token in ANY row.
                         The encoder, the cross-K/V prefill and the cross-attention then run on ceil32(bound) text positions
                         instead of max_seq_len: positions past the last token are padding whose keys carry zero weight and
                         whose rows nobody reads, so every valid position is bit-identical (SURVEY.md appendix A.3).
      reuse_encoder=False  reuse the encoder/cross-KV state left by the previous call (the caller guarantees the
                         encoder inputs are unchanged, e.g. generate.py's perplexity pass right after the answer pass)
    """

    def __init__(self, params, encoder, decoder):
        nn.Module.__init__(self)
        self.params = params
        self.encoder = encoder
        self.decoder = decoder
        self.vlfusion = VLFusion(encoder.config)
        self.config = {"encoder": encoder.config.to_dict(), "decoder": decoder.config.to_dict()}
        self._init_engine_state(params)
        self._calls = 0
        self._cls_start = None                # (tensor, version) last found to be all [CLS], see _decoder_prefix
        encoder._version = self._version      # one change counter for the whole model
        # plain attributes, not sub-modules: a registered back-reference would make the module tree cyclic
        object.__setattr__(encoder, "_owner", self)
        object.__setattr__(decoder, "_owner", self)

    # ---- engine plumbing --------------------------------------------------------------------------------------
    def _engine(self, device):
        return self._engine_for(device, self.encoder.config, self.decoder.config, "")

    def _score(self, eng, dec_input_ids, dec_attention_mask, dec_labels, loss_reduction, want_logits=True):
        if not dec_input_ids.is_contiguous() or dec_input_ids.dtype != torch.int64:
            raise ValueError("dec_input_ids must be a contiguous int64 tensor (it is modified in place like the reference does)")
        mode = self.params['mode']
        want_mean = ('train' in mode or 'eval' in mode) and loss_reduction
        # CrossEntropyLoss(ignore_index=0, reduction='mean') divides by the number of non-ignored targets and returns NaN when there
        # are none (models/visual_dialog_decoder.py:70-77).  The labels are the ids shifted left (:54-56), counted here BEFORE the
        # call replaces [SEP] by [PAD] in dec_input_ids in place.
        n = None
        if want_mean:
            n = (dec_input_ids[:, 1:] != 0).sum() if dec_labels is None else (dec_labels != 0).sum()
        loss, logits = eng.score(dec_input_ids, dec_attention_mask, dec_labels, want_logits=want_logits)
        if 'train' in mode or 'eval' in mode:
            if loss_reduction:
                loss = loss.sum() / n                    # 0 / 0 = NaN like the reference when every target is ignored
            else:
                loss = loss.reshape(-1)
        else:
            loss = None
        return Seq2SeqLMOutput(loss=loss, logits=logits)

    def forward(
        self,
        enc_image_features=None,
        enc_image_spatials=None,
        enc_image_mask=None,
        enc_image_target=None,
        enc_image_label=None,
        enc_next_sentence_labels=None,
        enc_input_ids=None,
        enc_segments=None,
        enc_sep_indices=None,
        enc_mlm_labels=None,
        enc_attention_mask=None,
        dec_input_ids=None,
        dec_attention_mask=None,
        dec_labels=None,
        loss_reduction=True,
        **decoding_kwargs
    ):
        eng = self._engine(enc_input_ids.device)
        B = enc_input_ids.shape[0]
        reuse = decoding_kwargs.get("reuse_encoder", False)
        decode = not ('train' in self.params['mode'] or 'eval' in self.params['mode'])
        ids_e, seg_e, att_e = enc_input_ids, enc_segments, enc_attention_mask
        if not reuse:
            hint = decoding_kwargs.get("enc_valid_len")
            if hint is not None:
                Lt = enc_input_ids.shape[1]
                Lt_eff = min(Lt, max(32, (int(hint) + 31) // 32 * 32))
                if Lt_eff < Lt:
                    ids_e, seg_e, att_e = ids_e[:, :Lt_eff], seg_e[:, :Lt_eff], (att_e[:, :Lt_eff] if att_e is not None else None)
        # decode mode, fresh encoder inputs: the whole call (encoder, fusion, cross-K/V prefill, 18 decode steps) is ONE graph replay
        whole_round = decode and not reuse and self.params.get("engine_round_graph", True) and enc_segments is not None
        if not reuse and not whole_round:
            enc = eng.encode(ids_e, enc_image_features, enc_image_spatials, seg_e, att_e, enc_image_mask)
            eng.prefill_cross(B, enc["Le"])

        if not decode:
            out = self._score(eng, dec_input_ids, dec_attention_mask, dec_labels, loss_reduction,
                              want_logits=decoding_kwargs.get("want_logits", True))
            return out.loss, out.logits

        # decode mode (models/visual_dialog_model.py:74-120): 18 new tokens after the caller's dec_input_ids, PAD after the first [SEP]
        self._check_decoder_start(dec_input_ids)
        self._calls += 1
        seed = decoding_kwargs.get("seed")
        if seed is None:
            # The reference draws independent torch.multinomial samples per call.  The device sampler is counter based, keyed by
            # (seed, global row, step): derive the seed from the run seed (options.py:43 -seed), the model's role (questioner and
            # teacher must not replay the same uniforms) and this model's call counter.  Callers that want draws that do not
            # depend on the batch / rank split pass seed= and row_offset= themselves (gst_visdial_b200/dialog.py does).
            seed = derive_seed(self.params.get("seed", 0), self.params.get("model", ""), self._calls)
        gen_kw = dict(
            num_beams=int(decoding_kwargs.get("num_beams", 1)),
            temperature=decoding_kwargs['temperature'],
            top_k=decoding_kwargs['top_k'],
            top_p=decoding_kwargs['top_p'],
            ngram_blocking_size=decoding_kwargs['ngram_blocking_size'],
            seed=seed,
            row_offset=int(decoding_kwargs.get("row_offset", 0)),
        )
        n_ret = int(decoding_kwargs.get("num_return_sequences", 1))
        if n_ret != 1:
            gen_kw["num_return_sequences"] = n_ret
        groups = int(decoding_kwargs.get("num_beam_groups", 1))
        penalty = float(decoding_kwargs.get("diversity_penalty", 0.0))
        if groups != 1 or penalty != 0.0:
            if groups > 1 and gen_kw["num_beams"] <= 1:
                raise ValueError(f"num_beam_groups = {groups} needs beam search (num_beams > 1)")
            gen_kw.update(num_beam_groups=groups, diversity_penalty=penalty)
        procs = dict(repetition_penalty=float(decoding_kwargs.get("repetition_penalty", 1.0)),
                     no_repeat_ngram_size=int(decoding_kwargs.get("no_repeat_ngram_size", 0)), min_length=int(decoding_kwargs.get("min_length", 0)))
        if procs != dict(repetition_penalty=1.0, no_repeat_ngram_size=0, min_length=0):
            gen_kw.update(procs)
        beam_args = dict(length_penalty=float(decoding_kwargs.get("length_penalty", 1.0)),
                         early_stopping=bool(decoding_kwargs.get("early_stopping", False)))
        if beam_args != dict(length_penalty=1.0, early_stopping=False):
            gen_kw.update(beam_args)
        if decoding_kwargs.get("bad_words_ids"):
            gen_kw["bad_words_ids"] = decoding_kwargs["bad_words_ids"]
        if decoding_kwargs.get("do_sample", False):
            if groups > 1:
                raise ValueError(f"num_beam_groups = {groups} cannot be combined with do_sample (beam sampling)")
            gen_kw["do_sample"] = True
        gen_kw["prefix"] = self._decoder_prefix(dec_input_ids, B, gen_kw["num_beams"], gen_kw["ngram_blocking_size"])
        if whole_round:
            # the n-gram blocking history is the (trimmed) encoder input itself: positions past the bound hold no token
            return eng.round(ids_e, enc_image_features, enc_image_spatials, seg_e, att_e, enc_image_mask, **gen_kw)
        return eng.generate(B, hist_ids=enc_input_ids, hist_segments=enc_segments, **gen_kw)

    def _check_decoder_start(self, dec_input_ids):
        """The reference continues from whatever prefix the caller passes (models/visual_dialog_model.py:86-110), and so does the
        engine (include/gstvd.h gstvd_generate, its prefix argument); its token bookkeeping needs the BERT bos / eos ids."""
        if dec_input_ids is None:
            return
        bos = int(getattr(self.decoder.config, "bos_token_id", 101) or 101)
        eos = int(getattr(self.decoder.config, "eos_token_id", 102) or 102)
        if bos != 101 or eos != 102:
            # the engine's token bookkeeping (start token, [SEP] -> [PAD] in the prefix, end of hypothesis) uses the BERT ids the
            # reference's configs carry (config/bert_base_6layer_6conect_dec.json: bos 101, eos 102)
            raise NotImplementedError(f"the engine decodes with bos_token_id 101 / eos_token_id 102; the decoder config says {bos} / {eos}")

    def _decoder_prefix(self, dec_input_ids, B, num_beams, ngram_blocking_size):
        """The decoder input the engine continues from: ``dec_input_ids`` [B, P], or None for one [CLS] per row.  None is only
        chosen where it changes the work: beam search with n-gram blocking skips the ban kernel of steps whose keys still hold a
        known [CLS] start, so a single-column all-[CLS] start is passed as None there (one host read per new tensor; the round loop
        passes the same tensor again).  Elsewhere the engine reads the start token on the device."""
        if dec_input_ids is None:
            return None
        if dec_input_ids.dim() != 2 or dec_input_ids.shape[0] != B:
            raise ValueError(f"dec_input_ids must be [B={B}, P], got {tuple(dec_input_ids.shape)}")
        if dec_input_ids.shape[1] == 1 and num_beams > 1 and ngram_blocking_size > 0:
            seen = self._cls_start
            if seen is not None and seen[0] is dec_input_ids and seen[1] == dec_input_ids._version:
                return None
            if bool((dec_input_ids == 101).all()):
                self._cls_start = (dec_input_ids, dec_input_ids._version)
                return None
        return dec_input_ids
