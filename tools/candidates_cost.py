"""Cost of several sequences per image (num_return_sequences = N): graph replays at the full config in bf16, B = 64 images with
150-token synthetic histories (tools/beam_ngram_cost.py:histories), every case alternating in one process.

    python tools/candidates_cost.py [--iters 20] [--json out.json]

Cases, each timed with CUDA events per round, medians over the rounds:
  * sample / sample_ngram4: top-k 7 sampling (temperature 0.7) without and with 4-gram blocking, N = 1 and N = 5 (N decode rows
    per image).  Every case runs as a call of T = 18 new tokens and as a call of T = 1; per-step time = (call(18) - call(1)) / 17;
  * beam5: beam-5 at N = 1 and N = 5 (the decode is the same, only the finalisation differs);
  * round: the answer half of one dialog round as generate_dialogs runs it with answer_candidates = N - one whole-round graph replay
    (encoder, cross-K/V prefill, 18 sampled steps with N candidates) followed by N perplexity passes (gstvd_score on B rows against
    the resident cross-K/V).
The GPU name and power limit are read in the same run and printed with the numbers.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch  # noqa: E402

from beam_ngram_cost import gpu_info, histories  # noqa: E402
from gst_visdial_b200 import weights as W  # noqa: E402
from gst_visdial_b200.engine import Engine  # noqa: E402

SAMPLE = dict(num_beams=1, temperature=0.7, top_k=7, top_p=0.0, seed=1)
MODES = {"sample": dict(SAMPLE, ngram_blocking_size=0), "sample_ngram4": dict(SAMPLE, ngram_blocking_size=4),
         "beam5": dict(num_beams=5)}
NS = (1, 5)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--hist", type=int, default=150)
    ap.add_argument("--iters", type=int, default=20, help="timed rounds; every round runs each case once")
    ap.add_argument("--json", default="", help="also write the result here")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    enc_cfg, dec_cfg = W.load_json_config(W.DEFAULT_ENC_CONFIG), W.load_json_config(W.DEFAULT_DEC_CONFIG)
    B, T = a.batch, 18
    eng = Engine(enc_cfg, dec_cfg, dtype="bf16", max_batch=B, max_beams=5)
    eng.load_state_dict(W.synthetic_state_dict(enc_cfg, dec_cfg, seed=0))
    b = {k: v.cuda() for k, v in histories(B, a.hist, enc_cfg.vocab_size, enc_cfg.v_feature_size).items()}
    rnd = (b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"], b["enc_image_mask"])
    hist = dict(hist_ids=b["enc_input_ids"], hist_segments=b["enc_segments"])

    def call(mode, N, steps):
        if mode == "round":
            out = eng.round(*rnd, num_return_sequences=N, max_new_tokens=steps, **MODES["sample"])
            for n in range(N):
                ids = out.view(B, N, -1)[:, n].contiguous()
                eng.score(ids, (ids != 0).float(), want_logits=False)
            return
        eng.generate(B, max_new_tokens=steps, num_return_sequences=N, **hist, **MODES[mode])

    cases = [(m, N, steps) for m in MODES for N in NS for steps in (T, 1)] + [("round", N, T) for N in NS]
    eng.round(*rnd, **MODES["sample"])                            # leaves the cross-K/V of the B images resident
    kernels = {}
    for c in cases:                                                # capture + warm up every graph
        for _ in range(3):
            call(*c)
        torch.cuda.synchronize()
        before = eng.launch_count
        call(*c)
        kernels[c] = eng.launch_count - before
    ev = {c: [] for c in cases}
    for _ in range(a.iters):
        for c in cases:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); call(*c); e1.record()
            ev[c].append((e0, e1))
    torch.cuda.synchronize()
    name, power = gpu_info()
    med = {c: sorted(e0.elapsed_time(e1) for e0, e1 in ev[c])[a.iters // 2] for c in cases}   # ms
    res = dict(gpu=name, power_limit=power, batch=B, hist_tokens=a.hist, new_tokens=T, iters=a.iters, modes=MODES, cases={})
    print(f"{name}, power limit {power}; B={B}, history {a.hist} tokens, {a.iters} alternating rounds, medians")
    for m in MODES:
        for N in NS:
            full, one = med[(m, N, T)], med[(m, N, 1)]
            r = dict(N=N, call_ms=full, call_t1_ms=one, us_per_step=1e3 * (full - one) / (T - 1), kernels_per_call=kernels[(m, N, T)])
            res["cases"][f"{m}_N{N}"] = r
            print(f"  {m:13s} N={N}: call {full:7.3f} ms, {r['us_per_step']:6.1f} us/step, {r['kernels_per_call']} kernels per call")
        r1, r5 = res["cases"][f"{m}_N1"], res["cases"][f"{m}_N{NS[-1]}"]
        res["cases"][f"{m}_ratio"] = dict(call=r5["call_ms"] / r1["call_ms"], step=r5["us_per_step"] / r1["us_per_step"])
        print(f"  {m:13s} N={NS[-1]} / N=1: call x{res['cases'][f'{m}_ratio']['call']:.3f}, step x{res['cases'][f'{m}_ratio']['step']:.3f}")
    for N in NS:
        r = dict(N=N, ms=med[("round", N, T)], kernels=kernels[("round", N, T)])
        res["cases"][f"round_N{N}"] = r
        print(f"  round (answer + {N} perplexity passes) N={N}: {r['ms']:7.3f} ms, {r['kernels']} kernels")
    ratio = med[("round", NS[-1], T)] / med[("round", 1, T)]
    res["cases"]["round_ratio"] = ratio
    print(f"  round N={NS[-1]} / N=1: x{ratio:.3f}")
    print(json.dumps(res))
    if a.json:
        with open(a.json, "w") as f:
            json.dump(res, f, indent=1)
    eng.close()


if __name__ == "__main__":
    main()
