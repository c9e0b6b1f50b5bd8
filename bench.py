#!/usr/bin/env python
"""bench.py - throughput of the generation hot path on N B200s of one node, BASELINE.json metric and configs.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload W] [--dump-outputs DIR]   # this framework (N > 1: torchrun)
    python bench.py --impl reference [--workload W] [...]                   # the reference's algorithm on the host CPU cores

Workloads (BASELINE.json `configs`; the default is configs[1], the configuration the metric is quoted on):
  gen_teacher  configs[1]  teacher enc_dec_a, beam-5 answer generation, batch 64 / GPU, 10 rounds, bf16.  One step = one batch of
                           64 complete 10-round dialogs: per round a synthetic 6-12 token question is spliced into the history
                           (generate.py:148-160), encoder + cross-KV prefill + 18 beam-search steps run, the answer is spliced
                           back (generate.py:214-228).  Unit: dialogs/s.
  gen_qa_ppl   configs[2]  questioner enc_dec_q (4-gram blocking) + teacher enc_dec_a alternating, temperature 0.7 / top-k 7
                           sampling like generate.py:138-141,177-180, plus the answer-perplexity pass (generate.py:183-209);
                           global batch 256 over 8 GPUs = 32 images / GPU.  Unit: dialogs/s.
  select_data  configs[3]  -select_data scoring: teacher-forced perplexity of (context, 18-token answer) pairs
                           (generate.py:183-209, dataloader_cc12m_gen.py:193-199), 256 pairs / GPU / step (BASELINE.json names no batch
                           for this config; 64 -> 256 raises the GEMM roofline from 0.55 to 0.78).  Unit: pairs/s.
  nsp_rank     configs[4]  enc_only_a discriminative ranking: 40 items x 100 candidate answers, every candidate its own
                           256-token encoder pass (evaluate_disc.py:66-83).  Unit: candidates/s.

Prints ONE JSON line (rank 0).  `value` = device-resident inputs; `e2e` = pinned host inputs copied in and results copied out
inside the timed region, through the reference-shaped module API.  `roofline` = the tcgen05 GEMM launches with M >= 1024 measured
live with CUDA events (tensor bound) and, in `entries`, the decode step timed with CUDA events around graph replays (HBM bound).
`cpu_baseline` times oracle/ (the CPU restatement of the reference) on a bounded sample on this host - bench.py is one of the
few places allowed to execute oracle/.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

WORKLOADS = ("gen_teacher", "gen_qa_ppl", "select_data", "nsp_rank")
# GFLOP per unit, SURVEY.md section 8d / BASELINE.md section 2 (2 M N K over the padded reference shapes, discarded heads excluded)
GF_ENCODER, GF_PREFILL, GF_DECODE_ROW, GF_SCORE18 = 76.66, 8.30, 4.61, 12.91


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="gen_teacher", choices=WORKLOADS)
    ap.add_argument("--batch", type=int, default=0, help="units per GPU per forward (0: the workload's configuration: 64 / 32 / 256 / 40)")
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--beams", type=int, default=5)
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--no-trim", action="store_true",
                    help="run the encoder on all 256 history positions instead of ceil32(longest history) (A/B aid; results are identical)")
    ap.add_argument("--streams", type=int, default=0,
                    help="independent batches in flight per GPU (each on its own CUDA stream and engine context); 1 = strictly serial; "
                         "0 = the workload's default (gen_teacher 2, gen_qa_ppl 3, the tensor-bound ones 1)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-budget-s", type=float, default=150.0, help="wall-clock cap of the reference arm")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the results of the last timed step (rank 0) as DIR/<name>.npy, float32 / float64, for comparing two builds")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.batch <= 0:
        a.batch = {"gen_teacher": 64, "gen_qa_ppl": 32, "select_data": 256, "nsp_rank": 40}[a.workload]
    if a.streams <= 0:
        a.streams = {"gen_teacher": 2, "gen_qa_ppl": 3}.get(a.workload, 1)      # measured: profiles/r2_scheduling_experiments.txt items 6, 10
    return a


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return d, "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


# ---------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i",
                                       str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(",") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for n, v in zip(names, r[4:8]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


# ---------------------------------------------------------------------------------------------------------------------
# Workload descriptions (names, units, FLOP counts) shared by both arms
def workload_info(a):
    w = a.workload
    if w == "gen_teacher":
        return dict(metric="synthetic dialogs/sec (10 rounds, beam 5)", unit="dialogs/s",
                    name=(f"configs[1]: teacher enc_dec_a beam-{a.beams} answer generation, batch {a.batch}/GPU, {a.rounds} rounds, {a.dtype}, "
                          f"36+1 x 2048 synthetic region feats, 18 new tokens/answer"),
                    tf_per_unit=a.rounds * (GF_ENCODER + GF_PREFILL + a.beams * GF_DECODE_ROW) / 1e3)
    if w == "gen_qa_ppl":
        return dict(metric="synthetic dialogs/sec (10 rounds, questioner + teacher + answer perplexity)", unit="dialogs/s",
                    name=(f"configs[2]: questioner enc_dec_q (4-gram blocking) + teacher enc_dec_a alternating {a.rounds}-round generation, "
                          f"temperature 0.7 / top-k 7 sampling, answer-perplexity pass, batch {a.batch}/GPU (global 256 on 8 GPUs), {a.dtype}"),
                    tf_per_unit=a.rounds * (2 * GF_ENCODER + 2 * GF_PREFILL + 2 * GF_DECODE_ROW + GF_SCORE18) / 1e3)
    if w == "select_data":
        return dict(metric="teacher-forced (context, answer) pairs scored/sec (-select_data perplexity)", unit="pairs/s",
                    name=(f"configs[3]: -select_data perplexity scoring of (context, 18-token answer) pairs, {a.batch} pairs/GPU/step, "
                          f"histories of 0-9 rounds, {a.dtype}"),
                    tf_per_unit=(GF_ENCODER + GF_SCORE18) / 1e3)
    return dict(metric="NSP-ranked answer candidates/sec (enc_only_a, 100 candidates per item)", unit="candidates/s",
                name=(f"configs[4]: enc_only_a discriminative ranking, {a.batch} items x 100 candidates per step "
                      f"(every candidate a 256-token encoder pass), histories of 1-10 rounds, {a.dtype}"),
                tf_per_unit=GF_ENCODER / 1e3)


# ---------------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's algorithm (oracle port) on a bounded sample of the same workload
def _cpu_setup(a, threads):
    from gst_visdial_b200 import weights as W
    torch.set_num_threads(threads)
    enc_cfg, dec_cfg = W.load_json_config(W.DEFAULT_ENC_CONFIG), W.load_json_config(W.DEFAULT_DEC_CONFIG)
    return enc_cfg, dec_cfg, W.synthetic_state_dict(enc_cfg, dec_cfg, seed=0)


def cpu_sample(a, state, images=1):
    """Runs the reference algorithm once on the workload's bounded sample; returns (seconds, units, description).
    No KV cache: the whole prefix and the cross-attention K/V are recomputed every step, and the discarded pre-training heads
    are evaluated like models/vilbert_dialog.py:1482 does - oracle/ over fp32, all host threads."""
    from gst_visdial_b200 import synthetic as S
    from oracle import beam as OB
    from oracle import restatement as R
    enc_cfg, dec_cfg, sd = state
    w = a.workload
    b = S.synthetic_batch(0, images, vocab_size=enc_cfg.vocab_size, v_feature_size=enc_cfg.v_feature_size)
    ids, seg = b["enc_input_ids"], b["enc_segments"]
    enc_len = (ids != 0).sum(-1)
    if w in ("gen_teacher", "gen_qa_ppl"):
        t0 = time.perf_counter()
        with torch.no_grad():
            if w == "gen_teacher":
                q = torch.stack([S.synthetic_utterance(i, 0, enc_cfg.vocab_size) for i in range(images)])
            else:
                q = R.generate_greedy_or_sample(sd, enc_cfg, dec_cfg, b, 0.7, 7, 0.0, 4, faithful_waste=True)
            R.splice(ids, seg, enc_len, q, None, set())
            b["enc_att_mask"] = (ids != 0).float()
            if w == "gen_teacher":
                seq_t, seq_v = R.encoder(sd, enc_cfg, ids, b["enc_image_feat"], b["enc_image_loc"], seg, b["enc_att_mask"], b["enc_image_mask"])
                R.wasted_heads(sd, seq_t, seq_v)
                OB.beam_search(sd, enc_cfg, dec_cfg, b, num_beams=a.beams, precomputed_encoder=(seq_t, seq_v))
            else:
                ans = R.generate_greedy_or_sample(sd, enc_cfg, dec_cfg, b, 0.7, 7, 0.0, 0, faithful_waste=True)
                R.score_answers(sd, enc_cfg, dec_cfg, b, ans, faithful_waste=True)
        dt = time.perf_counter() - t0
        return dt, images / a.rounds, (f"{images} image(s) x 1 round (of {a.rounds}; per-round work does not depend on the round index because "
                                       f"the reference pads the text to 256), fp32, scaled to a {a.rounds}-round dialog")
    if w == "select_data":
        ans = torch.stack([S.synthetic_utterance(i, 1, enc_cfg.vocab_size) for i in range(images)])
        t0 = time.perf_counter()
        with torch.no_grad():
            R.score_answers(sd, enc_cfg, dec_cfg, b, ans, faithful_waste=True)
        return time.perf_counter() - t0, images, f"{images} (context, answer) pair(s): encoder + discarded heads + teacher-forced decoder + CE, fp32"
    t0 = time.perf_counter()
    with torch.no_grad():
        seq_t, seq_v = R.encoder(sd, enc_cfg, ids, b["enc_image_feat"], b["enc_image_loc"], seg, b["enc_att_mask"], b["enc_image_mask"])
        R.wasted_heads(sd, seq_t, seq_v)
        R.nsp_scores(sd, seq_t, seq_v)
    return time.perf_counter() - t0, images, f"{images} candidate(s): encoder + discarded heads + poolers + NSP head, fp32"


def cpu_baseline_block(a, repeats=3, images=(1,)):
    threads = os.cpu_count() or 1
    state = _cpu_setup(a, threads)
    cpu_sample(a, state, images[0])                                   # warm-up
    out = None
    extra = {}
    for n in images:
        ts, units, desc = [], None, None
        for _ in range(repeats if n == images[0] else 1):     # the larger samples run once: the whole leg stays within ~2 minutes
            dt, units, desc = cpu_sample(a, state, n)
            ts.append(dt)
        v = units / statistics.mean(ts)
        if out is None:
            out = {"value": v, "unit": workload_info(a)["unit"], "cores": threads, "kind": "port",
                   "sample": f"{desc}; mean of {repeats} repeats = {statistics.mean(ts):.2f} s"}
        else:
            extra[f"value_batch{n}"] = v
    out.update(extra)
    return out


def run_reference(a, rank, world):
    """--impl reference: the reference's CPU path (oracle port; the Python reference cannot travel to this box)."""
    if rank != 0:
        return
    info = workload_info(a)
    threads = os.cpu_count() or 1
    state = _cpu_setup(a, threads)
    times, units, desc = [], 1.0, ""
    t_start, done_w = time.perf_counter(), 0
    for i in range(a.warmup + a.steps):
        dt, units, desc = cpu_sample(a, state, 1)
        over = (time.perf_counter() - t_start) > a.cpu_budget_s
        if i >= a.warmup or over:
            times.append(dt)
        else:
            done_w += 1
        if over and times:
            break
    t = statistics.mean(times)
    value = units / t
    line = {
        "impl": "reference", "metric": info["metric"], "value": value, "unit": info["unit"], "n_gpus": a.gpus, "steps": len(times),
        "warmup": done_w, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": {"workload": info["name"]},
        "cpu_baseline": {"value": value, "unit": info["unit"], "cores": threads, "kind": "port", "sample": f"{desc}; {len(times)} timed repeats"},
        "e2e": {"value": value, "unit": info["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    _emit(line)


# ---------------------------------------------------------------------------------------------------------------------
_REAL_STDOUT = None


def _quiet_stdout():
    """Everything that libraries print to fd 1 (e.g. NCCL's version banner) goes to stderr; the ONE JSON line is written to
    the original stdout by _emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def _emit(line):
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    if _REAL_STDOUT is None:
        os.write(1, data)
    else:
        os.write(_REAL_STDOUT, data)


def _checksum(t: torch.Tensor) -> int:
    """Position-weighted sum of an integer tensor (or of the raw bits of a float tensor): equal tensors <=> equal checksums in practice."""
    x = t.detach()
    if x.is_floating_point():
        x = x.float().contiguous().view(torch.int32)
    x = x.reshape(-1).to(torch.int64)
    w = torch.arange(1, x.numel() + 1, device=x.device, dtype=torch.int64)
    return int((x * w).sum().item() & 0x7FFFFFFFFFFFFFFF)


# ---------------------------------------------------------------------------------------------------------------------
# GPU arm: one "slot" = one in-flight batch = its own models / engine contexts / CUDA stream / inputs
def _build_enc_dec(params, sd, dev):
    from gst_visdial_b200.models.visual_dialog_decoder import VisualDialogDecoder
    from gst_visdial_b200.models.visual_dialog_encoder import VisualDialogEncoder
    from gst_visdial_b200.models.visual_dialog_model import EncoderDecoderModel
    enc, dec = VisualDialogEncoder(params), VisualDialogDecoder(params)
    dec.decoder.bert.embeddings = enc.bert_pretrained.bert.embeddings            # generate.py:65
    model = EncoderDecoderModel(params, enc, dec)
    model.load_state_dict(sd)
    model.to(dev).eval()
    return model


def make_slot(a, si, rank, world, dev, local, enc_cfg, dec_cfg, sds):
    from gst_visdial_b200 import synthetic as S
    from gst_visdial_b200 import weights as W
    B, w = a.batch, a.workload
    S_ = a.streams
    start = (rank * S_ + si) * B                       # weak scaling: every rank / stream owns its own images
    base = {"model_enc_config": W.DEFAULT_ENC_CONFIG, "model_dec_config": W.DEFAULT_DEC_CONFIG, "gpu_ids": [local], "mode": "cc12m_gen",
            "compute_dtype": a.dtype, "engine_max_batch": B, "engine_max_beams": max(a.beams, 1), "engine_flags": int(os.environ.get("GSTVD_ENGINE_FLAGS", "0")), "seed": 0}
    sl = dict(stream=torch.cuda.Stream(device=dev), start=start)
    vs, vf = enc_cfg.vocab_size, enc_cfg.v_feature_size
    if w in ("gen_teacher", "gen_qa_ppl"):
        sl["a_model"] = _build_enc_dec(dict(base, model="enc_dec_a"), sds["a"], dev)
        if w == "gen_qa_ppl":
            sl["q_model"] = _build_enc_dec(dict(base, model="enc_dec_q", engine_max_beams=1), sds["q"], dev)
        host = S.synthetic_batch(start, B, vocab_size=vs, v_feature_size=vf)
        host["questions"] = torch.stack([torch.stack([S.synthetic_utterance(start + i, r, vs) for r in range(a.rounds)]) for i in range(B)])
    elif w == "select_data":
        sl["a_model"] = _build_enc_dec(dict(base, model="enc_dec_a", engine_max_beams=1), sds["a"], dev)
        host = S.synthetic_history_batch(start, B, vocab_size=vs, v_feature_size=vf, rounds=[(start + i) % 10 for i in range(B)])
        host["answers"] = torch.stack([S.synthetic_utterance(start + i, 99, vs) for i in range(B)])
    else:
        from gst_visdial_b200.models.visual_dialog_encoder import VisualDialogEncoder
        chunk = 2000          # encoder passes per engine call: 500 -> 0.836 of the sustained bf16 rate, 1000 -> 0.855, 2000 -> 0.860 (same scores)
        p = dict(base, model="enc_only_a", mode="vd_eval_val", engine_max_batch=chunk)
        enc = VisualDialogEncoder(p)
        enc.load_state_dict({k[len("encoder."):]: v for k, v in sds["a"].items() if k.startswith("encoder.")})
        enc.to(dev).eval()
        sl["encoder"], sl["chunk"] = enc, chunk
        host = S.synthetic_candidate_batch(start, B, 100, vocab_size=vs, v_feature_size=vf)
    host = {k: v.pin_memory() for k, v in host.items()}
    sl["host"] = host
    sl["dev"] = {k: (v if k == "hist_len_bound" else v.to(dev)) for k, v in host.items()}      # the bound stays a host scalar
    if w in ("gen_teacher", "gen_qa_ppl"):
        # device-resident inputs: the caller keeps the (host-side) token counts the history bound is built from, like a loader that
        # knows its caption lengths - otherwise every dialog would start with a device read that drains the slot's stream
        sl["dev"]["enc_len_host"] = (host["enc_input_ids"] != 0).sum(-1).to(torch.int64)
        sl["dev"]["questions_len_host"] = (host["questions"] != 0).sum(-1).to(torch.int64)
    return sl


def slot_engines(sl, dev):
    out = []
    for k in ("a_model", "q_model"):
        if k in sl:
            out.append(sl[k]._engine(dev))
    if "encoder" in sl:
        out.append(sl["encoder"]._engine_for(dev, sl["encoder"].config, None, "encoder."))
    return out


def run_step(a, sl, dev, from_host, to_host):
    """One step of the workload on this slot's stream; returns the tuple of result tensors (device, or pinned host when to_host)."""
    from gst_visdial_b200 import ranking as RK
    from gst_visdial_b200.dialog import generate_dialogs
    w = a.workload
    src = sl["host"] if from_host else sl["dev"]
    with torch.cuda.stream(sl["stream"]):
        if w == "gen_teacher":
            akw = dict(temperature=1.0, top_k=1, top_p=0.0, ngram_blocking_size=0, num_beams=a.beams)
            res = generate_dialogs(sl["a_model"], src, questions=src["questions"], num_rounds=a.rounds, a_kwargs=akw, with_ppl=False, device=dev,
                                   trim_history=not a.no_trim, row_offset=sl["start"])
            outs = (res.answers, res.abnormal)
        elif w == "gen_qa_ppl":
            res = generate_dialogs(sl["a_model"], src, q_model=sl["q_model"], num_rounds=a.rounds, with_ppl=True, device=dev,
                                   trim_history=not a.no_trim, seed=0, row_offset=sl["start"])
            outs = (res.answers, res.abnormal, res.questions, res.answer_ppl)
        elif w == "select_data":
            batch = {k: v.to(dev, non_blocking=True) for k, v in src.items()} if from_host else src
            ppl = RK.answer_perplexity(sl["a_model"], batch, batch["answers"], device=dev, trim_history=not a.no_trim,
                                       hist_len_bound=int(sl["host"]["hist_len_bound"][0]))
            outs = (ppl,)
        else:
            scores = RK.nsp_rank_items(sl["encoder"], src, chunk=sl["chunk"], device=dev, trim_history=not a.no_trim)
            outs = (scores,)
        if to_host:                                     # device -> pinned host, asynchronous on this slot's stream
            if "out_host" not in sl:
                sl["out_host"] = [torch.empty(o.shape, dtype=o.dtype).pin_memory() for o in outs]
            for h, o in zip(sl["out_host"], outs):
                h.copy_(o, non_blocking=True)
            return tuple(sl["out_host"])
        return outs


# names of the tensors run_step returns, per workload
OUTPUT_NAMES = {"gen_teacher": ("answers", "abnormal"), "gen_qa_ppl": ("answers", "abnormal", "questions", "answer_ppl"),
                "select_data": ("answer_ppl",), "nsp_rank": ("nsp_scores",)}
DUMP_MAX_BYTES = 64 * 10**6


def dump_outputs(a, outs, out_dir):
    """Writes one step's results as <out_dir>/<name>.npy: floating-point results as float32, integer ones (token ids, flags) as
    float64, which holds them exactly.  Above DUMP_MAX_BYTES in all, a fixed seeded sample of rows (leading dimension, the same
    rows for every array) is written instead, with their indices as sample_rows.npy."""
    import numpy as np
    arrs = {n: o.detach().cpu().numpy().astype(np.float32 if o.is_floating_point() else np.float64)
            for n, o in zip(OUTPUT_NAMES[a.workload], outs)}
    total = sum(x.nbytes for x in arrs.values())
    rows = next(iter(arrs.values())).shape[0]
    if total > DUMP_MAX_BYTES:
        keep = max(1, rows * (DUMP_MAX_BYTES - 8 * rows) // total)         # 8 * rows: room for sample_rows
        idx = np.sort(np.random.default_rng(0).choice(rows, size=keep, replace=False))
        arrs = {n: x[idx] for n, x in arrs.items()}
        arrs["sample_rows"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for n, x in arrs.items():
        np.save(os.path.join(out_dir, f"{n}.npy"), x)


def h2d_bytes(a, sl):
    skip = ("image_id", "dec_att_mask", "hist_len_bound")
    return sum(v.numel() * v.element_size() for k, v in sl["host"].items() if k not in skip)


def decode_step_roofline(a, sl, dev, peaks, peak_src):
    """Second roofline entry: the KV-cached decode step (HBM bound), timed with CUDA events around graph replays of the 18-step
    generate call on the slot's stream, on the state the last timed dialog left resident (final-round history length)."""
    if a.workload not in ("gen_teacher", "gen_qa_ppl"):
        return None
    eng = sl["a_model"]._engine(dev)
    B = a.batch
    K = a.beams if a.workload == "gen_teacher" else 1
    kw = dict(num_beams=K) if K > 1 else dict(num_beams=1, temperature=0.7, top_k=7, seed=1)
    st = sl["stream"]
    T = eng.max_new_tokens
    with torch.cuda.stream(st):
        for _ in range(2):
            eng.generate(B, **kw)
        reps = 10
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        for _ in range(reps):
            eng.generate(B, **kw)
        e1.record(st)
        e1.synchronize()
        ms_step = e0.elapsed_time(e1) / (reps * T)
        geo = eng.decode_geometry(B)
        l0 = eng.launch_count
        eng.generate(B, **kw)
        geo["kernels_per_step"] = int(round((eng.launch_count - l0 - 3) / T))
    # algorithmic bytes of one step: every decoder matrix + the LM head once (bf16), each image's cross K/V up to its last
    # unmasked key once (shared by its beams), each row's self K/V history (mean over the 18 steps), fp32 logits not counted
    H, L, V, F = geo["hidden"], geo["layers"], geo["vocab"], geo["ffn"]
    w_bytes = 2.0 * (L * (4 * H * H + 2 * H * H + 2 * H * F) + V * H)          # qkv(3) + o + cross q + cross o = 6 H^2, FFN 2 H F
    cross_bytes = 2.0 * L * 2 * H * float(geo["cross_keys_total"])
    self_bytes = 2.0 * L * 2 * H * B * K * (T + 1) / 2.0
    total = w_bytes + cross_bytes + self_bytes
    peak = float(peaks.get("hbm_gbs", 6650.0))
    ach = total / (ms_step * 1e-3) / 1e9
    traffic = None                                  # dram read + write of one whole decode step from the committed ncu capture
    tp = os.path.join(ROOT, "profiles", "decode_step_traffic.json")
    if os.path.exists(tp):
        try:
            traffic = json.load(open(tp)).get("dram_bytes_per_step")
        except Exception:
            traffic = None
    return {"kernel": f"decode step ({geo['kernels_per_step']} kernels: 12 x [qkv GEMM, self-attention, o GEMM, cross-q GEMM, cross-attention, "
                      f"cross-o GEMM, FFN1, FFN2] + LM head + selection, CUDA-graph replay)",
            "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
            "peak_source": peak_src + ", hbm_gbs",
            "ms_per_decode_step": ms_step, "rows": B * K,
            "algorithmic_bytes_per_step": total,
            "bytes_breakdown": {"decoder_weights_and_lm_head": w_bytes, "cross_kv": cross_bytes, "self_kv": self_bytes},
            "measured_in": "CUDA events around 10 graph replays of the 18-step generate call, single stream, after the timed region"}


def main():
    _quiet_stdout()
    a = parse()
    from gst_visdial_b200 import dist as D
    if a.impl == "reference":
        run_reference(a, int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")))
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200; there is no CPU fallback (use --impl reference for the CPU arm)")
    rank, world, local = D.init_from_env("nccl")
    if world != a.gpus and world > 1:
        raise SystemExit(f"--gpus {a.gpus} but WORLD_SIZE={world}")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)

    from gst_visdial_b200 import weights as W
    info = workload_info(a)
    enc_cfg = W.load_json_config(W.DEFAULT_ENC_CONFIG)
    dec_cfg = W.load_json_config(W.DEFAULT_DEC_CONFIG)
    sds = {"a": W.synthetic_state_dict(enc_cfg, dec_cfg, seed=0)}
    if a.workload == "gen_qa_ppl":
        sds["q"] = W.synthetic_state_dict(enc_cfg, dec_cfg, seed=7)
    B = a.batch
    a.streams = S_ = max(1, min(a.streams, a.steps))
    units_per_step = B * (100 if a.workload == "nsp_rank" else 1)

    # One set of models (= engine contexts: weights, workspace, KV cache, graphs) and one CUDA stream per in-flight batch.
    # Decode steps are latency-bound chains of small kernels; independent batches on different streams fill the SMs those chains
    # leave idle.  Every forward call still sees the workload's batch.
    slots = [make_slot(a, si, rank, world, dev, local, enc_cfg, dec_cfg, sds) for si in range(S_)]
    engines = [e for sl in slots for e in slot_engines(sl, dev)]

    def barrier():
        # drain this rank's own queue BEFORE meeting the others: a rank with work still outstanding (rank 0 runs the decode-step
        # roofline pass alone) would otherwise leave the collective, wait for its own GPU and start its timed region late - the
        # other ranks then wait for it at the final all_gather and the max over ranks charges that skew to the step time
        torch.cuda.synchronize(dev)
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize(dev)

    host_ms = [0.0, 0.0]
    state = {"S": S_}

    def launches_total():
        return sum(e.launch_count for e in engines)

    def timed(from_host, to_host, steps, profile):
        S_now = state["S"]
        barrier()
        if profile:
            for e in engines:
                e.profile_gemm(True, 1024)
        l0 = launches_total()
        cur = torch.cuda.current_stream(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(cur)
        for sl in slots:
            sl["stream"].wait_event(e0)
        t_host, c_host = time.perf_counter(), time.process_time()
        # one submitting host thread per stream: a single thread blocks on the launch queue of one stream and starves the
        # others; the C ABI / torch calls release the GIL
        outs = [None] * S_now
        first = [None] * S_now

        def worker(si):
            torch.cuda.set_device(dev)
            for i in range(si, steps, S_now):
                outs[si] = run_step(a, slots[si], dev, from_host, to_host)
                if first[si] is None and not to_host:
                    with torch.cuda.stream(slots[si]["stream"]):          # the copy must be ordered after the step on ITS stream
                        first[si] = tuple(o.clone() for o in outs[si])

        if S_now == 1:
            worker(0)
        else:
            threads = [threading.Thread(target=worker, args=(si,)) for si in range(S_now)]
            for th in threads:
                th.start()
            for th in threads:
                th.join()
        gathered = None
        if world > 1:
            # The only collective of the job: ONE final all_gather (NCCL over NVLink) of this rank's last results per stream,
            # issued from the main thread after every stream has drained (collectives issued concurrently from several host
            # threads would not be ordered consistently across ranks).
            for sl in slots:
                cur.wait_stream(sl["stream"])
            mine = [o for o in outs if o is not None]
            cat = [torch.cat([o[j].to(dev) for o in mine], 0) for j in range(len(mine[0]))]
            gathered = D.gather_results(cat, [cat[0].shape[0]] * world)
        host_ms[0] = (time.perf_counter() - t_host) * 1e3 / steps      # wall time the submitting threads needed per step
        host_ms[1] = (time.process_time() - c_host) * 1e3 / steps      # CPU time (all threads of this process) per step
        for sl in slots:
            cur.wait_stream(sl["stream"])
        e1.record(cur)
        barrier()
        ms = e0.elapsed_time(e1)
        prof = None
        if profile:
            parts = [e.profile_read() for e in engines]
            prof = {k: sum(p_[k] for p_ in parts) for k in parts[0]}
            for e in engines:
                e.profile_gemm(False, 0)
        launches = launches_total() - l0
        t = torch.tensor([ms], device=dev)
        if world > 1:
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        return float(t.item()), launches, prof, outs, first, gathered

    n_warm = max(a.warmup, 3, S_)                      # every slot captures its decode graphs during warm-up
    for i in range(n_warm):
        run_step(a, slots[i % S_], dev, False, False)
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    ms, launches, prof, outs, first, _ = timed(False, False, a.steps, False)
    host_issue_ms, host_cpu_ms = host_ms[0], host_ms[1]
    clocks = sampler.stop() if sampler else None
    if a.dump_outputs and rank == 0:
        dump_outputs(a, outs[(a.steps - 1) % S_], a.dump_outputs)      # step i ran on slot i % S_
    # ---- self-check of the timed outputs (a silent garbage path must not print a number) ----
    out0 = outs[0]
    check = {"ids_checksum": _checksum(out0[0]), "finite": True, "in_range": True, "deterministic": None, "varied": True}
    for o in out0:
        if o.is_floating_point():
            fin = torch.isfinite(o) | torch.isnan(o) if a.workload == "gen_qa_ppl" else torch.isfinite(o)   # ppl of an answer that is only [SEP] is NaN by contract
            check["finite"] = check["finite"] and bool(fin.all())
    if a.workload.startswith("gen_"):
        ids = out0[0]
        check["in_range"] = bool(((ids >= 0) & (ids < enc_cfg.vocab_size)).all())
        check["varied"] = int(ids.unique().numel()) > 8
    if first[0] is not None and a.steps > S_:
        # the same slot ran the same batch (and the same sampling seeds) several times: identical results expected - the kernels are
        # deterministic by construction (fixed reduction orders, no floating-point atomics)
        check["deterministic"] = all(torch.equal(torch.nan_to_num(x.float()), torch.nan_to_num(y.float())) for x, y in zip(first[0], out0))
    if not (check["finite"] and check["in_range"] and check["varied"] and check["deterministic"] is not False):
        raise SystemExit(f"bench.py: output self-check failed: {check}")
    cs_path = os.path.join(ROOT, "profiles", "bench_checksums.json")
    key = f"{a.workload}/{a.dtype}/b{B}/k{a.beams}/r{a.rounds}" + ("/notrim" if a.no_trim else "")
    check["expected"] = None
    if os.path.exists(cs_path):
        try:
            check["expected"] = json.load(open(cs_path)).get(key)
        except Exception:
            pass
    check["matches_recorded"] = None if check["expected"] is None else (check["expected"] == check["ids_checksum"])
    check["key"] = key

    # The roofline of the GEMM kernel is taken from a separate, strictly serial pass (one stream) over the same workload: with
    # several batches in flight the event pairs around one stream's GEMMs would also span other streams' kernels, and while the
    # per-launch events are recorded the engine launches eagerly (events cannot be recorded inside the whole-round graph), which
    # must not be part of the timed region.
    state["S"] = 1
    serial_steps = max(2, min(a.steps, 4))
    ms_serial, _, prof, _, _, _ = timed(False, False, serial_steps, True)
    prof = dict(prof); prof["serial_pass_steps"] = serial_steps; prof["serial_ms_per_step"] = ms_serial / serial_steps
    state["S"] = S_
    peaks, peak_src = measured_peaks()
    decode_entry = decode_step_roofline(a, slots[0], dev, peaks, peak_src) if rank == 0 else None
    for i in range(S_):
        run_step(a, slots[i], dev, True, True)
    ms_e2e, _, _, outs_h, _, _ = timed(True, True, a.steps, False)

    if rank == 0:
        n_units = units_per_step * world * a.steps
        value = n_units / (ms / 1e3)
        e2e = n_units / (ms_e2e / 1e3)
        h2d = h2d_bytes(a, slots[0])
        d2h = sum(o.numel() * o.element_size() for o in outs_h[0])
        peak_tf = float(peaks.get("bf16_tflops_sustained", 1400.0))
        ach_tf = prof["flops"] / (prof["ms"] * 1e-3) / 1e12 if prof and prof["ms"] > 0 else None
        traffic = None
        tp = os.path.join(ROOT, "profiles", "gemm_traffic.json")
        if os.path.exists(tp):
            try:
                traffic = json.load(open(tp)).get("dram_bytes_per_launch")
            except Exception:
                traffic = None
        gemm_entry = {"kernel": "gemm_tc_kernel (tcgen05 GEMM, launches with M >= 1024: encoder, cross-KV prefill, teacher-forced decoder)",
                      "bound": "tensor", "achieved": ach_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": (ach_tf / peak_tf) if ach_tf else None,
                      "traffic": traffic, "peak_source": peak_src + ", bf16_tflops_sustained (kernel timed inside a long step)",
                      "launches": prof["launches"] if prof else 0,
                      "kernel_ms_per_step": prof["ms"] / prof.get("serial_pass_steps", a.steps) if prof else None,
                      "measured_in": "serial single-stream pass inside this run (eager launches, one CUDA event pair per GEMM)",
                      "algorithmic_flops_per_launch": prof["flops"] / max(prof["launches"], 1) if prof else None}
        roofline = dict(gemm_entry)
        roofline["entries"] = [gemm_entry] + ([decode_entry] if decode_entry else [])
        line = {
            "metric": info["metric"], "value": value, "unit": info["unit"], "n_gpus": world, "steps": a.steps, "warmup": n_warm,
            "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": a.dtype,
            "data": "synthetic",
            "config": {"workload": info["name"], "workload_key": a.workload, "global_batch": B * world, "rounds": a.rounds, "beams": a.beams,
                       "parallelism": f"dp{world}: independent image shards, one final NCCL all_gather of the results",
                       "history_positions": "all 256" if a.no_trim else "ceil32(longest history in the batch): padded positions are never read, results identical",
                       "streams_per_gpu": S_, "batch_per_forward": B, "units_per_step_per_gpu": units_per_step,
                       "host_enqueue_ms_per_step": host_issue_ms, "host_cpu_ms_per_step": host_cpu_ms,
                       "serial_eager_profiled_ms_per_step": prof.get("serial_ms_per_step") if prof else None,
                       "l2": "no explicit flush: each step streams >1.5 GB (0.78 GB bf16 weights per model, cross-KV, activations), "
                             "far beyond the 126 MB L2",
                       "end_to_end_tflops": value * info["tf_per_unit"], "tf_per_unit": info["tf_per_unit"],
                       "output_check": check},
            "clocks": clocks,
            "e2e": {"value": e2e, "unit": info["unit"], "h2d_bytes_per_step": int(h2d * world), "d2h_bytes_per_step": int(d2h * world),
                    "ms_per_step": ms_e2e / a.steps},
            "gpu_launches": int(launches),
            "roofline": roofline,
        }
        if world == 1 and not a.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_block(a, repeats=3, images=(1, 8) if a.workload == "gen_teacher" else (1,))
        _emit(line)
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
