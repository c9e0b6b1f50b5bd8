"""Cost of beam sampling (num_beams > 1 with do_sample): graph replays of the 18-step generate call at the full config in bf16 with
B = 64 images and 150-token synthetic histories (tools/beam_ngram_cost.histories), every case alternating in one process.

    python tools/beam_sample_cost.py [--iters 30] [--json out.json] [--txt out.txt]

Cases, without and with 4-gram blocking:
  * beam5: beam search with K = 5;
  * beam_sample5: beam sampling with K = 5, temperature 0.7, top-k 7;
  * beam_sample4x2: beam sampling with K = 4 and N = 2 searches per image (512 decode rows: still the deferred-LayerNorm path, M <= 512).
Per case: the device time of one generate call (CUDA events; the call also holds the beam init / finalize kernels and, with blocking,
the copy of the history into the graph's buffers) divided by its 18 decode steps, and the kernels per call (gstvd_launch_count).
Also the answer half of a dialog round as generate_dialogs runs it with -answer_candidates 2 -num_beams 4 -beam_sample: one whole-round
graph replay (encoder, cross-K/V prefill, 18 beam-sampled steps over N = 2 searches) and two perplexity passes, next to the same round
with beam search (K = 4, the 2 best beams).  The GPU name and power limit are read in the same run and printed with the numbers.
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

WARP = dict(temperature=0.7, top_k=7, top_p=0.0, seed=1)
MODES = {"beam5": dict(num_beams=5), "beam_sample5": dict(num_beams=5, do_sample=True, **WARP),
         "beam_sample4x2": dict(num_beams=4, do_sample=True, num_return_sequences=2, **WARP)}
ROUNDS = {"round_beam4_best2": dict(num_beams=4, num_return_sequences=2),
          "round_beam_sample4x2": dict(num_beams=4, do_sample=True, num_return_sequences=2, **WARP)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--hist", type=int, default=150)
    ap.add_argument("--iters", type=int, default=30, help="timed calls per case (alternating)")
    ap.add_argument("--json", default="", help="also write the result here")
    ap.add_argument("--txt", default="", help="also write the printed summary here")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    enc_cfg, dec_cfg = W.load_json_config(W.DEFAULT_ENC_CONFIG), W.load_json_config(W.DEFAULT_DEC_CONFIG)
    B, T = a.batch, 18
    eng = Engine(enc_cfg, dec_cfg, dtype="bf16", max_batch=B, max_beams=8)
    eng.load_state_dict(W.synthetic_state_dict(enc_cfg, dec_cfg, seed=0))
    b = {k: v.cuda() for k, v in histories(B, a.hist, enc_cfg.vocab_size, enc_cfg.v_feature_size).items()}
    rnd = (b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"], b["enc_image_mask"])
    hist = dict(hist_ids=b["enc_input_ids"], hist_segments=b["enc_segments"])

    def call(case):
        mode, n = case
        if mode in ROUNDS:
            kw = ROUNDS[mode]
            N = kw["num_return_sequences"]
            out = eng.round(*rnd, **kw)
            for i in range(N):
                ids = out.view(B, N, -1)[:, i].contiguous()
                eng.score(ids, (ids != 0).float(), want_logits=False)
            return
        eng.generate(B, ngram_blocking_size=n, **hist, **MODES[mode])

    cases = [(m, n) for n in (0, 4) for m in MODES] + [(m, 0) for m in ROUNDS]
    eng.round(*rnd, **MODES["beam5"])                             # leaves the cross-K/V of the B images resident
    kernels = {}
    for c in cases:                                                # capture + warm up every graph
        for _ in range(3):
            call(c)
        torch.cuda.synchronize()
        before = eng.launch_count
        call(c)
        kernels[c] = eng.launch_count - before
    times = {c: [] for c in cases}
    for _ in range(a.iters):
        for c in cases:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); call(c); e1.record()
            times[c].append((e0, e1))
    torch.cuda.synchronize()
    name, power = gpu_info()
    res = dict(gpu=name, power_limit=power, batch=B, hist_tokens=a.hist, steps=T, iters=a.iters, modes=MODES, rounds=ROUNDS, cases={})
    lines = [f"{name}, power limit {power}; full config bf16, B={B}, history {a.hist} tokens, {a.iters} alternating graph replays per case"]
    ms = {c: sorted(e0.elapsed_time(e1) for e0, e1 in times[c]) for c in cases}
    for c in cases:
        mode, n = c
        m = ms[c]
        med = m[len(m) // 2]
        if mode in ROUNDS:
            r = dict(ms_median=med, ms_min=m[0], ms_max=m[-1], kernels=kernels[c])
            res["cases"][mode] = r
            lines.append(f"  {mode} (answer half of a round, 2 perplexity passes): {med:.3f} ms (median; min {m[0]:.3f}, max {m[-1]:.3f}), "
                         f"{kernels[c]} kernels")
            continue
        base = ms[("beam5", n)][len(m) // 2]
        r = dict(mode=mode, ngram=n, us_per_step_median=1e3 * med / T, us_per_step_min=1e3 * m[0] / T, us_per_step_max=1e3 * m[-1] / T,
                 kernels_per_call=kernels[c], vs_beam5_pct=100.0 * (med / base - 1.0))
        res["cases"][f"{mode}_n{n}"] = r
        lines.append(f"  {mode} n={n}: {r['us_per_step_median']:.1f} us/step (median; min {r['us_per_step_min']:.1f}, max "
                     f"{r['us_per_step_max']:.1f}), {r['kernels_per_call']} kernels per call, {r['vs_beam5_pct']:+.2f} % vs beam5")
    text = "\n".join(lines)
    print(text)
    print(json.dumps(res))
    if a.json:
        with open(a.json, "w") as f:
            json.dump(res, f, indent=1)
    if a.txt:
        with open(a.txt, "w") as f:
            f.write(text + "\n")
    eng.close()


if __name__ == "__main__":
    main()
