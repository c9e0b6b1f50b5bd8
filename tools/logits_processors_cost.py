"""Cost of the logits processors (repetition_penalty, no_repeat_ngram_size, min_length): graph replays of the 18-step generate call at the
full config in bf16 with B = 64 images and 150-token synthetic histories (tools/beam_ngram_cost.histories), every case alternating in one
process.

    python tools/logits_processors_cost.py [--iters 30] [--json out.json] [--txt out.txt]

Two decode setups: top-k 7 sampling (temperature 0.7) with 4-gram question blocking, as the questioner runs, and beam-5 search.  For each,
five processor settings: off, each processor alone (repetition_penalty 1.3, no_repeat_ngram_size 3, min_length 8) and all three.  Per case:
the device time of one generate call (CUDA events) divided by its 18 decode steps, the kernels per call (gstvd_launch_count), and the
change against the processors-off case of the same setup.  The GPU name and power limit are read in the same run.
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

SETUPS = {"sample_topk7_ngram4": dict(temperature=0.7, top_k=7, top_p=0.0, seed=1, ngram_blocking_size=4),
          "beam5": dict(num_beams=5)}
PROCS = {"off": {}, "repetition_penalty": dict(repetition_penalty=1.3), "no_repeat_ngram": dict(no_repeat_ngram_size=3),
         "min_length": dict(min_length=8), "all_three": dict(repetition_penalty=1.3, no_repeat_ngram_size=3, min_length=8)}


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
        setup, procs = case
        eng.generate(B, **hist, **SETUPS[setup], **PROCS[procs])

    cases = [(s, p) for s in SETUPS for p in PROCS]
    eng.round(*rnd, num_beams=5)                                  # leaves the cross-K/V of the B images resident
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
    res = dict(gpu=name, power_limit=power, batch=B, hist_tokens=a.hist, steps=T, iters=a.iters, setups=SETUPS, processors=PROCS, cases={})
    lines = [f"{name}, power limit {power}; full config bf16, B={B}, history {a.hist} tokens, {a.iters} alternating graph replays per case"]
    ms = {c: sorted(e0.elapsed_time(e1) for e0, e1 in times[c]) for c in cases}
    for c in cases:
        setup, procs = c
        m = ms[c]
        med = m[len(m) // 2]
        base = ms[(setup, "off")][len(m) // 2]
        r = dict(setup=setup, processors=procs, us_per_step_median=1e3 * med / T, us_per_step_min=1e3 * m[0] / T,
                 us_per_step_max=1e3 * m[-1] / T, kernels_per_call=kernels[c], vs_off_pct=100.0 * (med / base - 1.0))
        res["cases"][f"{setup}_{procs}"] = r
        lines.append(f"  {setup} {procs}: {r['us_per_step_median']:.1f} us/step (median; min {r['us_per_step_min']:.1f}, max "
                     f"{r['us_per_step_max']:.1f}), {r['kernels_per_call']} kernels per call, {r['vs_off_pct']:+.2f} % vs off")
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
