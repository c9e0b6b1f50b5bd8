"""Cost of diverse beam search (beam groups with a Hamming diversity penalty): graph replays of the 18-step generate call with
K = 6 beams in G = 1, 3 and 6 groups (penalty 0.5 for G > 1), without and with 4-gram blocking, alternating in one process, at the
full config in bf16 with B = 64 images and 150-token synthetic histories (tools/beam_ngram_cost.histories).

    python tools/group_beam_cost.py [--iters 30] [--json out.json] [--txt out.txt]

Prints, per case, the device time of one generate call (CUDA events; the call also holds the beam init / finalize kernels and, with
blocking, the copy of the history into the graph's buffers) divided by its 18 decode steps, and the kernels per call counted by
gstvd_launch_count.  The GPU name and power limit are printed with the numbers.
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--beams", type=int, default=6)
    ap.add_argument("--groups", default="1,3,6")
    ap.add_argument("--penalty", type=float, default=0.5)
    ap.add_argument("--hist", type=int, default=150)
    ap.add_argument("--iters", type=int, default=30, help="timed calls per case (alternating)")
    ap.add_argument("--json", default="", help="also write the result here")
    ap.add_argument("--txt", default="", help="also write the printed summary here")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    enc_cfg, dec_cfg = W.load_json_config(W.DEFAULT_ENC_CONFIG), W.load_json_config(W.DEFAULT_DEC_CONFIG)
    B, K, T = a.batch, a.beams, 18
    eng = Engine(enc_cfg, dec_cfg, dtype="bf16", max_batch=B, max_beams=K)
    eng.load_state_dict(W.synthetic_state_dict(enc_cfg, dec_cfg, seed=0))
    b = {k: v.cuda() for k, v in histories(B, a.hist, enc_cfg.vocab_size, enc_cfg.v_feature_size).items()}
    out = eng.encode(b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"], b["enc_image_mask"])
    eng.prefill_cross(B, out["Le"])
    cases = [(int(g), n) for n in (0, 4) for g in a.groups.split(",")]

    def call(case):
        G, n = case
        return eng.generate(B, num_beams=K, num_beam_groups=G, diversity_penalty=a.penalty if G > 1 else 0.0, ngram_blocking_size=n,
                            hist_ids=b["enc_input_ids"], hist_segments=b["enc_segments"])

    kernels = {}
    for c in cases:                                                # capture + warm up every graph
        for _ in range(3):
            call(c)
        torch.cuda.synchronize()
        before = eng.launch_count
        call(c)
        kernels[c] = eng.launch_count - before
    times = {c: [] for c in cases}
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.iters * len(cases))]
    for i in range(a.iters):
        for j, c in enumerate(cases):
            e0, e1 = ev[i * len(cases) + j]
            e0.record(); call(c); e1.record()
            times[c].append((e0, e1))
    torch.cuda.synchronize()
    name, power = gpu_info()
    res = dict(gpu=name, power_limit=power, batch=B, beams=K, penalty=a.penalty, hist_tokens=a.hist, steps=T, iters=a.iters, cases={})
    lines = [f"{name}, power limit {power}; full config bf16, B={B} K={K} history {a.hist} tokens, penalty {a.penalty} for G > 1, "
             f"{a.iters} alternating graph replays of the {T}-step call per case"]
    for c in cases:
        G, n = c
        ms = sorted(e0.elapsed_time(e1) for e0, e1 in times[c])
        med = ms[len(ms) // 2]
        base = sorted(e0.elapsed_time(e1) for e0, e1 in times[(1, n)])[len(ms) // 2]
        r = dict(groups=G, ngram=n, us_per_step_median=1e3 * med / T, us_per_step_min=1e3 * ms[0] / T, us_per_step_max=1e3 * ms[-1] / T,
                 kernels_per_call=kernels[c], vs_one_group_pct=100.0 * (med / base - 1.0))
        res["cases"][f"G{G}_n{n}"] = r
        lines.append(f"  G={G} n={n}: {r['us_per_step_median']:.1f} us/step (median; min {r['us_per_step_min']:.1f}, max "
                     f"{r['us_per_step_max']:.1f}), {r['kernels_per_call']} kernels per call, {r['vs_one_group_pct']:+.2f} % vs G=1")
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
