"""Python wrapper of one gstvd context (one per process and device).

PyTorch is only plumbing here: it owns the device tensors and the stream; every computation happens in
libgstvd.so through the C ABI of include/gstvd.h.
"""
from __future__ import annotations

import ctypes
from typing import Mapping, Optional

import torch

from . import _lib
from ._lib import (GSTVD_BF16, GSTVD_F32, GSTVD_SELECT_BEAM, GSTVD_SELECT_BEAM_SAMPLE, GSTVD_SELECT_SAMPLE, GstvdConfig, GstvdError,
                   GstvdGenParams, check)

DTYPES = {"fp32": GSTVD_F32, "float32": GSTVD_F32, "f32": GSTVD_F32, torch.float32: GSTVD_F32,
          "bf16": GSTVD_BF16, "bfloat16": GSTVD_BF16, torch.bfloat16: GSTVD_BF16}


def _select_mode(num_beams, do_sample):
    """HF generate()'s choice: beams with do_sample = beam sampling, beams without = beam search, one beam = the sampler."""
    if num_beams > 1:
        return GSTVD_SELECT_BEAM_SAMPLE if do_sample else GSTVD_SELECT_BEAM
    return GSTVD_SELECT_SAMPLE


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def bad_words_array(bad_words_ids):
    """HF-style ``bad_words_ids`` (a list of id lists) as the int32 array gstvd_gen_params.bad_words_ids points to: the sequences
    concatenated, each closed by -1.  None or [] gives None."""
    if not bad_words_ids:
        return None
    flat = []
    for seq in bad_words_ids:
        flat.extend(int(w) for w in seq)
        flat.append(-1)
    return (ctypes.c_int32 * len(flat))(*flat)


_KERNEL_NAMES = {v: k for k, v in _lib.GEMM_KERNELS.items()}
_STORE_NAMES = {v: k for k, v in _lib.GEMM_STORES.items()}


def _variant_names(ran):
    """(kernel, store) names of the int32 pair a GEMM op entry reports."""
    return _KERNEL_NAMES.get(ran[0]), _STORE_NAMES.get(ran[1])


class Engine:
    """Owns a gstvd_ctx.  ``dec_cfg=None`` builds an encoder-only context (enc_only_a / NSP ranking)."""

    def __init__(self, enc_cfg, dec_cfg=None, device=0, dtype="bf16", max_batch=64, max_beams=5, max_text_len=256,
                 max_regions=37, max_new_tokens=18, max_dec_len=25, flags=0):
        if not torch.cuda.is_available():
            raise RuntimeError("gst_visdial_b200.Engine needs a CUDA device (sm_100); there is no CPU fallback")
        self.lib = _lib.load()
        self.device = torch.device("cuda", device if isinstance(device, int) else torch.device(device).index or 0)
        self.enc_cfg, self.dec_cfg = enc_cfg, dec_cfg
        self.dtype = DTYPES[dtype]
        c = GstvdConfig()
        c.abi_version = _lib.GSTVD_ABI_VERSION
        c.compute_dtype = self.dtype
        for f in ("vocab_size", "hidden_size", "num_hidden_layers", "num_attention_heads", "intermediate_size",
                  "max_position_embeddings", "type_vocab_size", "v_feature_size", "v_hidden_size", "v_num_hidden_layers",
                  "v_num_attention_heads", "v_intermediate_size", "bi_hidden_size", "bi_num_attention_heads"):
            setattr(c, f, int(getattr(enc_cfg, f)))
        vb, tb = list(enc_cfg.v_biattention_id), list(enc_cfg.t_biattention_id)
        if len(vb) != len(tb) or len(vb) > _lib.GSTVD_MAX_CONNECTIONS:
            raise ValueError("v_biattention_id / t_biattention_id must have equal length <= 16")
        c.num_connections = len(vb)
        for i, (a, b) in enumerate(zip(vb, tb)):
            c.v_biattention_id[i] = int(a)
            c.t_biattention_id[i] = int(b)
        if dec_cfg is not None:
            if dec_cfg.hidden_size != enc_cfg.hidden_size or dec_cfg.vocab_size != enc_cfg.vocab_size:
                raise ValueError("decoder hidden/vocab size must match the encoder (shared embeddings)")
            c.dec_num_hidden_layers = int(dec_cfg.num_hidden_layers)
            c.dec_num_attention_heads = int(dec_cfg.num_attention_heads)
            c.dec_intermediate_size = int(dec_cfg.intermediate_size)
        c.max_batch, c.max_text_len, c.max_regions = int(max_batch), int(max_text_len), int(max_regions)
        c.max_new_tokens, c.max_beams, c.max_dec_len, c.flags = int(max_new_tokens), int(max_beams), int(max_dec_len), int(flags)
        self.cfg = c
        self.max_batch, self.max_beams, self.max_new_tokens = int(max_batch), int(max_beams), int(max_new_tokens)
        ctx = ctypes.c_void_p()
        rc = self.lib.gstvd_create(ctypes.byref(c), self.device.index, ctypes.byref(ctx))
        if rc < 0:
            check(None, rc)
        self.ctx = ctx
        self.weights_loaded = False

    # ---- lifecycle ------------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "ctx", None):
            self.lib.gstvd_destroy(self.ctx)
            self.ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _dev(self, t: Optional[torch.Tensor], dtype) -> Optional[torch.Tensor]:
        if t is None:
            return None
        if t.device != self.device or t.dtype != dtype or not t.is_contiguous():
            t = t.to(device=self.device, dtype=dtype, non_blocking=True).contiguous()
        return t

    @property
    def launch_count(self) -> int:
        return int(self.lib.gstvd_launch_count(self.ctx))

    def decode_geometry(self, B=None):
        """Measurement aid: the sizes bench.py's decode-step roofline is computed from, for the resident cross K/V of ``B`` images."""
        d = self.dec_cfg
        out = dict(hidden=int(d.hidden_size), layers=int(d.num_hidden_layers), vocab=int(d.vocab_size), ffn=int(d.intermediate_size))
        B = int(B or self.max_batch)
        counts = torch.empty(B, dtype=torch.int32, device=self.device)
        check(self.ctx, self.lib.gstvd_cross_key_counts(self.ctx, B, _ptr(counts), self._stream()))
        out["cross_keys_total"] = int(counts.sum().item())
        return out

    def profile_gemm(self, enable: bool, min_rows: int = 0):
        check(self.ctx, self.lib.gstvd_profile_gemm(self.ctx, int(enable), int(min_rows)))

    def profile_read(self):
        f, b, ms, n = ctypes.c_double(), ctypes.c_double(), ctypes.c_double(), ctypes.c_int64()
        check(self.ctx, self.lib.gstvd_profile_read(self.ctx, ctypes.byref(f), ctypes.byref(b), ctypes.byref(ms), ctypes.byref(n)))
        return dict(flops=f.value, bytes=b.value, ms=ms.value, launches=n.value)

    # ---- weights --------------------------------------------------------------------------------------------
    def load_state_dict(self, sd: Mapping[str, torch.Tensor], prefix: str = "", strict: bool = True):
        """``sd`` uses EncoderDecoderModel key names after ``prefix`` is prepended (e.g. prefix='encoder.' for a bare
        VisualDialogEncoder.state_dict())."""
        stream = self._stream()
        keep = []
        for name, t in sd.items():
            t32 = t.detach()
            if t32.dtype != torch.float32 or not t32.is_contiguous():
                t32 = t32.float().contiguous()
            keep.append(t32)
            rc = self.lib.gstvd_load_weight(self.ctx, (prefix + name).encode(), _ptr(t32), t32.numel(), stream)
            if rc < 0:
                if not strict and rc == -1:
                    continue
                check(self.ctx, rc)
        if any(not k.is_cuda for k in keep):
            torch.cuda.synchronize(self.device)          # pageable host sources must outlive the async copies
        missing = self.lib.gstvd_missing_weights(self.ctx)
        if strict and missing:
            raise GstvdError(-1, f"{missing} expected weight tensors were not provided")
        check(self.ctx, self.lib.gstvd_finalize_weights(self.ctx, stream))
        self.weights_loaded = True
        del keep

    # ---- encoder --------------------------------------------------------------------------------------------
    def encode(self, input_ids, image_feat, image_loc, token_type_ids=None, attention_mask=None, image_mask=None,
               want_t=False, want_v=False, want_fused=False, want_nsp=False):
        ids = self._dev(input_ids, torch.int64)
        B, Lt = ids.shape
        feat = self._dev(image_feat, torch.float32)
        Lv = feat.shape[1]
        loc = self._dev(image_loc, torch.float32)
        seg = self._dev(token_type_ids, torch.int64)
        att = self._dev(attention_mask, torch.float32)
        imask = self._dev(image_mask, torch.float32)
        H, Hv = self.cfg.hidden_size, self.cfg.v_hidden_size
        f32 = dict(device=self.device, dtype=torch.float32)
        out = {}
        out_t = torch.empty(B, Lt, H, **f32) if want_t else None
        out_v = torch.empty(B, Lv, Hv, **f32) if want_v else None
        out_f = torch.empty(B, Lv + Lt, H, **f32) if want_fused else None
        out_fm = torch.empty(B, Lv + Lt, **f32) if want_fused else None
        out_nsp = torch.empty(B, 2, **f32) if want_nsp else None
        check(self.ctx, self.lib.gstvd_encode(self.ctx, B, Lt, Lv, _ptr(ids), _ptr(seg), _ptr(att), _ptr(feat), _ptr(loc),
                                              _ptr(imask), _ptr(out_t), _ptr(out_v), _ptr(out_f), _ptr(out_fm), _ptr(out_nsp),
                                              self._stream()))
        out.update(seq_t=out_t, seq_v=out_v, fused=out_f, fused_mask=out_fm, nsp=out_nsp, B=B, Le=Lv + Lt)
        return out

    # ---- decoder --------------------------------------------------------------------------------------------
    def prefill_cross(self, B, Le, enc_hidden=None, enc_mask=None):
        h = self._dev(enc_hidden, torch.float32)
        m = self._dev(enc_mask, torch.float32)
        check(self.ctx, self.lib.gstvd_prefill_cross(self.ctx, B, Le, _ptr(h), _ptr(m), self._stream()))

    def _prefix(self, prefix, B):
        """(device int64 [B, P] tensor or None, P) of a decoder prefix argument; None stands for one [CLS] per row.  A negative id
        ends a row's prefix (rows of different lengths, include/gstvd.h gstvd_generate); a row cannot start with one, which is
        checked here for a host tensor (a device tensor is not read on the host)."""
        if prefix is None:
            return None, 1
        if isinstance(prefix, torch.Tensor) and prefix.device.type == "cpu" and prefix.dim() == 2 and prefix.shape[1] > 0:
            bad = (prefix[:, 0] < 0).nonzero().flatten()
            if len(bad):
                raise ValueError(f"prefix row {int(bad[0])} starts with a negative id: every row needs at least one token")
        pre = self._dev(prefix, torch.int64)
        if pre.dim() != 2 or pre.shape[0] != B:
            raise ValueError(f"prefix must be [B={B}, P], got {tuple(pre.shape)}")
        return pre, pre.shape[1]

    def _gen_params(self, num_beams=1, temperature=1.0, top_k=1, top_p=0.0, ngram_blocking_size=0, seed=0, max_new_tokens=None,
                    row_offset=0, num_return_sequences=1, num_beam_groups=1, diversity_penalty=0.0, do_sample=False,
                    repetition_penalty=1.0, no_repeat_ngram_size=0, min_length=0, length_penalty=1.0, early_stopping=False, bad_words_ids=None):
        """The gstvd_gen_params of one decode request (include/gstvd.h gstvd_generate).  The bad-word array stays referenced by the
        returned struct (attribute ``_bad_words``) for as long as the struct lives."""
        gp = GstvdGenParams()
        gp.mode = _select_mode(num_beams, do_sample)
        gp.num_beams = int(num_beams)
        gp.max_new_tokens = int(max_new_tokens or self.max_new_tokens)
        gp.top_k, gp.temperature, gp.top_p = int(top_k), float(temperature), float(top_p)
        gp.ngram_blocking_size, gp.seed = int(ngram_blocking_size), int(seed) & (2**64 - 1)
        gp.row_offset = int(row_offset)
        gp.num_return_sequences, gp.num_beam_groups = int(num_return_sequences), int(num_beam_groups)
        gp.diversity_penalty = float(diversity_penalty)
        gp.repetition_penalty, gp.no_repeat_ngram_size, gp.min_length = float(repetition_penalty), int(no_repeat_ngram_size), int(min_length)
        gp.length_penalty, gp.early_stopping = float(length_penalty), int(early_stopping)
        gp._bad_words = bad_words_array(bad_words_ids)
        gp.bad_words_ids = ctypes.addressof(gp._bad_words) if gp._bad_words is not None else 0
        gp.bad_words_len = len(gp._bad_words) if gp._bad_words is not None else 0
        return gp

    def generate(self, B, num_beams=1, temperature=1.0, top_k=1, top_p=0.0, ngram_blocking_size=0, seed=0,
                 max_new_tokens=None, hist_ids=None, hist_segments=None, want_scores=False, row_offset=0, prefix=None,
                 num_return_sequences=1, num_beam_groups=1, diversity_penalty=0.0, do_sample=False, repetition_penalty=1.0,
                 no_repeat_ngram_size=0, min_length=0, length_penalty=1.0, early_stopping=False, bad_words_ids=None):
        """``row_offset``: global index of row 0; the sampler is keyed by (seed, row_offset + row, step), so an image draws the
        same tokens whichever batch or rank it lands in.  ``prefix``: int64 [B, P] decoder input to continue from (the reference's
        dec_input_ids), None = one [CLS] per row; the result holds the new tokens only.
        ``num_return_sequences`` = N: [B*N, T] image-major - the N best beams, or N sampled candidates per image of which
        candidate n draws like an N = 1 call with seed ``candidate_seed(seed, n)``.
        ``num_beam_groups`` = G > 1 with ``diversity_penalty``: diverse beam search, the K beams in G groups of K / G with a Hamming
        penalty between groups (contract in oracle/beam_groups.py).
        ``do_sample`` with ``num_beams`` > 1: beam sampling (HF beam_sample) with ``temperature`` / ``top_k`` / ``top_p`` / ``seed``;
        ``num_return_sequences`` = N then runs N independent searches per image, search n seeded ``candidate_seed(seed, n)``, and
        returns the best hypothesis of each (GSTVD_SELECT_BEAM_SAMPLE, contract in oracle/beam_sample.py).  With ``num_beams`` = 1
        the sampler runs whatever ``do_sample`` says.
        ``repetition_penalty`` (1 = off) / ``no_repeat_ngram_size`` (0 = off) / ``min_length`` (0 = off): HF's logits processors on each
        row's own decoder input, prefix included (contract in oracle/processors.py).
        ``length_penalty`` (1 = HF default) / ``early_stopping``: the beam modes' hypothesis scores sum / len ** length_penalty and
        is_done (contract in oracle/decode_args.py).  ``bad_words_ids``: HF-style list of id lists that the output never completes, in
        every mode.  The whole contract is at gstvd_generate in include/gstvd.h."""
        gp = self._gen_params(num_beams, temperature, top_k, top_p, ngram_blocking_size, seed, max_new_tokens, row_offset,
                              num_return_sequences, num_beam_groups, diversity_penalty, do_sample, repetition_penalty,
                              no_repeat_ngram_size, min_length, length_penalty, early_stopping, bad_words_ids)
        hid = self._dev(hist_ids, torch.int64) if ngram_blocking_size > 0 else None
        hseg = self._dev(hist_segments, torch.int64) if ngram_blocking_size > 0 else None
        Lh = hid.shape[1] if hid is not None else 0
        pre, P = self._prefix(prefix, B)
        N = gp.num_return_sequences
        out = torch.empty(B * max(N, 1), gp.max_new_tokens, device=self.device, dtype=torch.int64)
        scores = torch.empty(B * max(N, 1), device=self.device, dtype=torch.float32) if want_scores else None
        check(self.ctx, self.lib.gstvd_generate(self.ctx, B, ctypes.byref(gp), _ptr(pre), P, _ptr(hid), _ptr(hseg), Lh, _ptr(out),
                                                _ptr(scores), self._stream()))
        return (out, scores) if want_scores else out

    def round(self, input_ids, image_feat, image_loc, token_type_ids=None, attention_mask=None, image_mask=None, num_beams=1,
              temperature=1.0, top_k=1, top_p=0.0, ngram_blocking_size=0, seed=0, max_new_tokens=None, want_scores=False, row_offset=0,
              prefix=None, num_return_sequences=1, num_beam_groups=1, diversity_penalty=0.0, do_sample=False, repetition_penalty=1.0,
              no_repeat_ngram_size=0, min_length=0, length_penalty=1.0, early_stopping=False, bad_words_ids=None):
        """encode + prefill_cross + generate of one forward call as ONE graph replay (gstvd_round); the n-gram blocking history is
        ``input_ids`` / ``token_type_ids``.  Leaves the encoder / cross-K/V state resident like the three separate calls.
        ``prefix`` / ``num_return_sequences`` / ``num_beam_groups`` / ``diversity_penalty`` / ``do_sample`` / ``repetition_penalty`` /
        ``no_repeat_ngram_size`` / ``min_length`` / ``length_penalty`` / ``early_stopping`` / ``bad_words_ids``: as in ``generate``."""
        ids = self._dev(input_ids, torch.int64)
        B, Lt = ids.shape
        feat = self._dev(image_feat, torch.float32)
        Lv = feat.shape[1]
        loc = self._dev(image_loc, torch.float32)
        seg = self._dev(token_type_ids, torch.int64)
        att = self._dev(attention_mask, torch.float32)
        imask = self._dev(image_mask, torch.float32)
        gp = self._gen_params(num_beams, temperature, top_k, top_p, ngram_blocking_size, seed, max_new_tokens, row_offset,
                              num_return_sequences, num_beam_groups, diversity_penalty, do_sample, repetition_penalty,
                              no_repeat_ngram_size, min_length, length_penalty, early_stopping, bad_words_ids)
        pre, P = self._prefix(prefix, B)
        N = gp.num_return_sequences
        out = torch.empty(B * max(N, 1), gp.max_new_tokens, device=self.device, dtype=torch.int64)
        scores = torch.empty(B * max(N, 1), device=self.device, dtype=torch.float32) if want_scores else None
        check(self.ctx, self.lib.gstvd_round(self.ctx, B, Lt, Lv, _ptr(ids), _ptr(seg), _ptr(att), _ptr(feat), _ptr(loc), _ptr(imask),
                                             ctypes.byref(gp), _ptr(pre), P, _ptr(out), _ptr(scores), self._stream()))
        return (out, scores) if want_scores else out

    def score(self, dec_ids, dec_mask=None, labels=None, want_logits=False, want_loss=True, options_per_image=1):
        """``dec_ids`` (int64, on the engine's device, contiguous) is mutated in place when ``labels`` is None.
        ``options_per_image`` > 1: rows are option-major per image and share the image's cross-attention K/V."""
        if dec_ids.device != self.device or dec_ids.dtype != torch.int64 or not dec_ids.is_contiguous():
            raise ValueError("score: dec_ids must be a contiguous int64 tensor on the engine's device (it is updated in place)")
        B, L = dec_ids.shape
        m = self._dev(dec_mask, torch.float32)
        lab = self._dev(labels, torch.int64)
        V = self.cfg.vocab_size
        loss = torch.empty(B, L, device=self.device, dtype=torch.float32) if want_loss else None
        logits = torch.empty(B, L, V, device=self.device, dtype=torch.float32) if want_logits else None
        if options_per_image > 1:
            check(self.ctx, self.lib.gstvd_score_options(self.ctx, B // options_per_image, int(options_per_image), L, _ptr(dec_ids), _ptr(m),
                                                         _ptr(lab), _ptr(loss), _ptr(logits), self._stream()))
        else:
            check(self.ctx, self.lib.gstvd_score(self.ctx, B, L, _ptr(dec_ids), _ptr(m), _ptr(lab), _ptr(loss), _ptr(logits), self._stream()))
        return loss, logits

    def reorder_cache(self, beam_idx: torch.Tensor, length: int):
        bi = self._dev(beam_idx, torch.int32)
        B, K = bi.shape
        check(self.ctx, self.lib.gstvd_reorder_cache(self.ctx, B, K, int(length), _ptr(bi), self._stream()))

    def splice(self, enc_input_ids, enc_segments, attention_mask, enc_len, utt, segment_value=-1, strip_sep=False, abnormal=None):
        """In-place history append (generate.py:145-160 / :214-228).  All tensors must already live on the device."""
        B, Lt = enc_input_ids.shape
        u = self._dev(utt, torch.int64)
        check(self.ctx, self.lib.gstvd_splice(self.ctx, B, Lt, u.shape[1], _ptr(enc_input_ids), _ptr(enc_segments), _ptr(attention_mask),
                                              _ptr(enc_len), _ptr(u), int(segment_value), int(bool(strip_sep)), _ptr(abnormal),
                                              self._stream()))

    # ---- single operators (parity tests) ----------------------------------------------------------------------
    def op_linear(self, a, w, bias=None, act=0, dtype=None, out_dtype="fp32", ldc=None, hm=None, kernel=None, store=None, out=None,
                  want_variant=False):
        """One GEMM launch (gstvd_op_linear): act(a w^T + bias) from fp32 ``a`` [M, K], ``w`` [N, K].  ``out_dtype``: what the kernel
        stores (returned as fp32).  ``ldc``: row stride of the result (default N).  ``hm`` = (D, L, G, B): the head-major K/V layout of
        the cross-attention prefill, result [N / (D * G)][B][G][L][D].  ``kernel`` / ``store``: a name of _lib.GEMM_KERNELS /
        GEMM_STORES to force, None = the engine's choice.  ``out``: fp32 buffer holding the whole output region (M * ldc, or M * N
        head-major) whose elements the kernel does not store are kept; default NaN.  ``want_variant``: also return the
        (kernel, store) names that ran."""
        a, w = self._dev(a, torch.float32), self._dev(w, torch.float32)
        b = self._dev(bias, torch.float32)
        M, K = a.shape
        N = w.shape[0]
        ld = N if ldc is None else int(ldc)
        if out is None:
            shape = (N // (hm[0] * hm[2]), hm[3], hm[2], hm[1], hm[0]) if hm is not None else (M, ld)
            out = torch.full(shape, float("nan"), device=self.device, dtype=torch.float32)
        hm_arr = (ctypes.c_int32 * 4)(*[int(x) for x in hm]) if hm is not None else None
        ran = (ctypes.c_int32 * 2)(-1, -1)
        check(self.ctx, self.lib.gstvd_op_linear(self.ctx, self.dtype if dtype is None else DTYPES[dtype], M, N, K, _ptr(a), _ptr(w),
                                                 _ptr(b), int(act), _ptr(out), 0 if hm is not None else ld, DTYPES[out_dtype], hm_arr,
                                                 -1 if kernel is None else _lib.GEMM_KERNELS[kernel],
                                                 -1 if store is None else _lib.GEMM_STORES[store], ran, self._stream()))
        if hm is None and ldc is None:
            out = out.view(M, N)
        return (out, _variant_names(ran)) if want_variant else out

    def op_linear_ln(self, a, w, bias=None, a_stats=None, ln_gamma=None, ln_beta=None, res=None, res_stats=None, res_gamma=None,
                     res_beta=None, act=0, want_stats=False, kernel=None):
        """One deferred-LayerNorm GEMM launch (gstvd_op_linear_ln), fp32 tensors in and out: act(LN(a) w^T + bias + R) stored bf16.
        ``a_stats`` [K/32, M, 2]: per-32-column (mean, M2) of a's rows, with ``ln_gamma`` / ``ln_beta``: a's rows are LayerNormed
        through folded weights.  ``res`` [M, N]: raw residual, or with ``res_stats`` [N/32, M, 2] / ``res_gamma`` / ``res_beta`` its
        LayerNorm.  Returns (out [M, N], stats_out [N/32, M, 2] or None, (kernel, store) names)."""
        f = lambda t: self._dev(t, torch.float32)
        a, w, bias, a_stats, ln_gamma, ln_beta, res, res_stats, res_gamma, res_beta = map(
            f, (a, w, bias, a_stats, ln_gamma, ln_beta, res, res_stats, res_gamma, res_beta))
        M, K = a.shape
        N = w.shape[0]
        out = torch.empty(M, N, device=self.device, dtype=torch.float32)
        st = torch.full((N // 32, M, 2), float("nan"), device=self.device, dtype=torch.float32) if want_stats else None
        ran = (ctypes.c_int32 * 2)(-1, -1)
        check(self.ctx, self.lib.gstvd_op_linear_ln(self.ctx, M, N, K, _ptr(a), _ptr(a_stats), _ptr(ln_gamma), _ptr(ln_beta), _ptr(w),
                                                    _ptr(bias), _ptr(res), _ptr(res_stats), _ptr(res_gamma), _ptr(res_beta), int(act),
                                                    _ptr(out), _ptr(st), -1 if kernel is None else _lib.GEMM_KERNELS[kernel], ran,
                                                    self._stream()))
        return out, st, _variant_names(ran)

    def debug_cross_cache(self, B, Le):
        """The cross-attention K/V of the last prefill_cross, fp32 [layers, B, 2 * heads, Le, D] (k heads, then v heads)."""
        d = self.dec_cfg
        heads = int(d.num_attention_heads)
        buf = torch.empty(int(d.num_hidden_layers), B, 2 * heads, Le, int(d.hidden_size) // heads, dtype=torch.float32, device=self.device)
        check(self.ctx, self.lib.gstvd_debug_cross_cache(self.ctx, int(B), int(Le), _ptr(buf), self._stream()))
        return buf

    def op_add_layernorm(self, x, residual, gamma, beta, dtype=None):
        x = self._dev(x, torch.float32)
        r = self._dev(residual, torch.float32)
        g, b = self._dev(gamma, torch.float32), self._dev(beta, torch.float32)
        rows, width = x.shape
        y = torch.empty_like(x)
        check(self.ctx, self.lib.gstvd_op_add_layernorm(self.ctx, self.dtype if dtype is None else DTYPES[dtype], rows, width, _ptr(x),
                                                        _ptr(r), _ptr(g), _ptr(b), _ptr(y), self._stream()))
        return y

    def op_deferred_ln_chain(self, a1, w1, b1, res0, gamma1, beta1, w2, b2, gamma2, beta2, want_x1=False):
        """LN2(LN1(x1) w2^T + b2 + LN1(x1)) with x1 = a1 w1^T + b1 + res0, through the decode step's deferred-LayerNorm GEMM
        epilogues (no LayerNorm kernel between the two GEMMs).  bf16 contexts; fp32 tensors in and out."""
        f = lambda t: self._dev(t, torch.float32)
        a1, w1, b1, res0, gamma1, beta1, w2, b2, gamma2, beta2 = map(f, (a1, w1, b1, res0, gamma1, beta1, w2, b2, gamma2, beta2))
        M, K1 = a1.shape
        N = w1.shape[0]
        assert w1.shape == (N, K1) and w2.shape == (N, N) and res0.shape == (M, N)
        out = torch.empty(M, N, dtype=torch.float32, device=self.device)
        x1 = torch.empty(M, N, dtype=torch.float32, device=self.device) if want_x1 else None
        check(self.ctx, self.lib.gstvd_op_deferred_ln_chain(self.ctx, M, N, K1, _ptr(a1), _ptr(w1), _ptr(b1), _ptr(res0), _ptr(gamma1),
                                                            _ptr(beta1), _ptr(w2), _ptr(b2), _ptr(gamma2), _ptr(beta2), _ptr(out), _ptr(x1),
                                                            self._stream()))
        return (out, x1) if want_x1 else out

    def debug_self_cache(self, B, K, layer, kv, values=None):
        """Test access to the self-attention KV cache of one (layer, kv) in the (B, K) layout: fp32 [B, max_new_tokens, K, hidden].
        ``values`` given: written into the cache; else the current content is returned."""
        H = self.cfg.hidden_size
        if values is not None:
            buf = self._dev(values, torch.float32)
            assert buf.shape == (B, self.max_new_tokens, K, H)
            check(self.ctx, self.lib.gstvd_debug_self_cache(self.ctx, 1, B, K, layer, kv, _ptr(buf), self._stream()))
            torch.cuda.current_stream(self.device).synchronize()
            return None
        buf = torch.empty(B, self.max_new_tokens, K, H, dtype=torch.float32, device=self.device)
        check(self.ctx, self.lib.gstvd_debug_self_cache(self.ctx, 0, B, K, layer, kv, _ptr(buf), self._stream()))
        return buf

    def op_attention(self, q, k, v, heads, mask=None, neg=-10000.0, causal=False, dtype=None):
        q, k, v = self._dev(q, torch.float32), self._dev(k, torch.float32), self._dev(v, torch.float32)
        m = self._dev(mask, torch.float32)
        B, Lq, W = q.shape
        Lk = k.shape[1]
        out = torch.empty_like(q)
        check(self.ctx, self.lib.gstvd_op_attention(self.ctx, self.dtype if dtype is None else DTYPES[dtype], B, heads, Lq, Lk, W // heads,
                                                    _ptr(q), _ptr(k), _ptr(v), _ptr(m), float(neg), int(bool(causal)), _ptr(out),
                                                    self._stream()))
        return out

    SELF_KERNELS = {"default": -1, "first": 0, "v2": 1}
    CROSS_KERNELS = {"default": -1, "warp_tma": 0, "cta_tma": 1, "mma": 2, "simt": 3, "generic": 4}

    def op_dec_self_attn(self, qkv, cache, heads, P0=0, step=0, step_known=True, prefix_qkv=None, anc=None, kernel="default", dtype=None,
                         p0s=None):
        """One decode-step self-attention launch (include/gstvd.h gstvd_op_dec_self_attn) on fp32 ``qkv`` [B*K, 3H] and ``cache``
        [2, B, T, K, H]; ``anc`` uint8 [B*K, 32 or 64]; ``p0s`` int [B]: each image's own P0 (<= ``P0``), None = ``P0`` for all.
        Returns (out [B*K, H], the cache after the call); ``cache`` is not modified."""
        q = self._dev(qkv, torch.float32)
        c = self._dev(cache, torch.float32).clone()
        _, B, T, K, H = c.shape
        pre = self._dev(prefix_qkv, torch.float32)
        a = self._dev(anc, torch.uint8)
        p0 = self._dev(p0s, torch.int32)
        out = torch.empty(B * K, H, device=self.device, dtype=torch.float32)
        check(self.ctx, self.lib.gstvd_op_dec_self_attn(self.ctx, self.dtype if dtype is None else DTYPES[dtype], self.SELF_KERNELS[kernel], B, K,
                                                        int(heads), H // heads, T, int(P0), _ptr(p0), int(step), int(bool(step_known)), _ptr(q),
                                                        _ptr(pre), _ptr(c), _ptr(a), _ptr(out), self._stream()))
        return out, c

    def op_dec_cross_attn(self, q, cross_kv, K, mask=None, use_cross_len=True, kernel="default", dtype=None):
        """One decode-step cross-attention launch (gstvd_op_dec_cross_attn): fp32 ``q`` [B*K, H], ``cross_kv`` [B, 2*heads, Le, D],
        ``mask`` [B, Le].  Returns (out [B*K, H], cross_len int32 [B] or None)."""
        qd, kv, m = self._dev(q, torch.float32), self._dev(cross_kv, torch.float32), self._dev(mask, torch.float32)
        B, two_heads, Le, D = kv.shape
        cl = torch.empty(B, device=self.device, dtype=torch.int32) if use_cross_len else None
        out = torch.empty(qd.shape[0], qd.shape[1], device=self.device, dtype=torch.float32)
        check(self.ctx, self.lib.gstvd_op_dec_cross_attn(self.ctx, self.dtype if dtype is None else DTYPES[dtype], self.CROSS_KERNELS[kernel], B,
                                                         int(K), two_heads // 2, D, Le, _ptr(qd), _ptr(kv), _ptr(m), int(bool(use_cross_len)),
                                                         _ptr(cl), _ptr(out), self._stream()))
        return out, cl

    def op_anc_update(self, anc, beam_idx, T, P0, step, p0s=None):
        """One ancestry-table update (gstvd_op_anc_update): returns the updated copy of uint8 ``anc`` [B*K, 32 or 64].  ``p0s`` int [B]:
        each image's own P0 (<= ``P0``), None = ``P0`` for all."""
        bi = self._dev(beam_idx, torch.int32)
        B, K = bi.shape
        a = self._dev(anc, torch.uint8).clone()
        p0 = self._dev(p0s, torch.int32)
        check(self.ctx, self.lib.gstvd_op_anc_update(self.ctx, B, K, int(T), int(P0), _ptr(p0), int(step), _ptr(bi), _ptr(a), self._stream()))
        return a

    def op_beam_begin(self, B, K, max_new):
        check(self.ctx, self.lib.gstvd_op_beam_begin(self.ctx, B, K, max_new, self._stream()))
        self._beam_shape = (B, K)

    def op_beam_step(self, logits):
        lg = self._dev(logits, torch.float32)
        B, K = self._beam_shape
        bi = torch.empty(B, K, device=self.device, dtype=torch.int32)
        bt = torch.empty(B, K, device=self.device, dtype=torch.int32)
        bs = torch.empty(B, K, device=self.device, dtype=torch.float32)
        check(self.ctx, self.lib.gstvd_op_beam_step(self.ctx, _ptr(lg), lg.stride(0), _ptr(bi), _ptr(bt), _ptr(bs), self._stream()))
        return bi, bt, bs

    def op_beam_end(self, max_new):
        B, _ = self._beam_shape
        out = torch.empty(B, max_new, device=self.device, dtype=torch.int64)
        sc = torch.empty(B, device=self.device, dtype=torch.float32)
        check(self.ctx, self.lib.gstvd_op_beam_end(self.ctx, _ptr(out), _ptr(sc), self._stream()))
        return out, sc

    def op_sample(self, logits, step, temperature=1.0, top_k=1, top_p=0.0, ngram_blocking_size=0, seed=0, hist_ids=None,
                  hist_segments=None, prefix=None, row_offset=0, repetition_penalty=1.0, no_repeat_ngram_size=0, min_length=0,
                  bad_words_ids=None):
        """One sampling step on caller logits; ``prefix`` [rows, step + 1] is each row's decoder input so far, which n-gram blocking and
        the logits processors (``bad_words_ids`` included) read."""
        lg = self._dev(logits, torch.float32)
        gp = self._gen_params(temperature=temperature, top_k=top_k, top_p=top_p, ngram_blocking_size=ngram_blocking_size, seed=seed,
                              row_offset=row_offset, repetition_penalty=repetition_penalty, no_repeat_ngram_size=no_repeat_ngram_size,
                              min_length=min_length, bad_words_ids=bad_words_ids)
        hid, hseg, pre = self._dev(hist_ids, torch.int64), self._dev(hist_segments, torch.int64), self._dev(prefix, torch.int64)
        rows = lg.shape[0]
        out = torch.empty(rows, device=self.device, dtype=torch.int32)
        check(self.ctx, self.lib.gstvd_op_sample(self.ctx, rows, _ptr(lg), lg.stride(0), ctypes.byref(gp), _ptr(hid), _ptr(hseg),
                                                 hid.shape[1] if hid is not None else 0, _ptr(pre),
                                                 pre.shape[1] if pre is not None else 0, int(step), _ptr(out), self._stream()))
        return out
