"""Cost of question-history n-gram blocking in beam mode: graph replays of the 18-step generate call with n = 0 and n = 4,
alternating in one process, at the full config in bf16 with B = 64 images, K = 5 beams and 150-token synthetic histories
(caption, then alternating questions - segment 0, the history the blocking reads - and answers - segment 1).

    python tools/beam_ngram_cost.py [--iters 40] [--json out.json]

Prints, per n, the device time of one generate call (CUDA events; the call also holds the beam init / finalize kernels and, for
n > 0, the copy of the history into the graph's buffers) divided by its 18 decode steps, and the kernels per step counted by
gstvd_launch_count.  The GPU name and power limit are printed with the numbers.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from gst_visdial_b200 import synthetic as S, weights as W  # noqa: E402
from gst_visdial_b200.engine import Engine  # noqa: E402


def histories(B, length, vocab_size, v_feature_size):
    b = S.synthetic_batch(0, B, vocab_size=vocab_size, v_feature_size=v_feature_size)
    ids, seg = b["enc_input_ids"], b["enc_segments"]
    for i in range(B):
        pos, rnd = int((ids[i] != 0).sum()), 0
        while pos < length:
            u = S.synthetic_utterance(i, rnd, vocab_size)
            u = u[u != 0][: length - pos]
            ids[i, pos:pos + len(u)] = u
            seg[i, pos:pos + len(u)] = rnd % 2                    # questions 0, answers 1
            pos += len(u); rnd += 1
    Lt = (length + 31) // 32 * 32
    b["enc_input_ids"], b["enc_segments"] = ids[:, :Lt].contiguous(), seg[:, :Lt].contiguous()
    b["enc_att_mask"] = (b["enc_input_ids"] != 0).float()
    return b


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [x.strip() for x in q.split(",")]
    except Exception:                                               # noqa: BLE001 - the numbers stand without it
        name, power = torch.cuda.get_device_name(), "unknown"
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--beams", type=int, default=5)
    ap.add_argument("--hist", type=int, default=150)
    ap.add_argument("--iters", type=int, default=40, help="timed calls per n (alternating)")
    ap.add_argument("--json", default="", help="also write the result here")
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
    ns = (0, 4)

    def call(n):
        return eng.generate(B, num_beams=K, ngram_blocking_size=n, hist_ids=b["enc_input_ids"], hist_segments=b["enc_segments"])

    kernels = {}
    for n in ns:                                                   # capture + warm up every graph
        for _ in range(3):
            call(n)
        torch.cuda.synchronize()
        before = eng.launch_count
        call(n)
        kernels[n] = eng.launch_count - before
    times = {n: [] for n in ns}
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.iters * len(ns))]
    for i in range(a.iters):
        for j, n in enumerate(ns):
            e0, e1 = ev[i * len(ns) + j]
            e0.record(); call(n); e1.record()
            times[n].append((e0, e1))
    torch.cuda.synchronize()
    name, power = gpu_info()
    res = dict(gpu=name, power_limit=power, batch=B, beams=K, hist_tokens=a.hist, steps=T, iters=a.iters)
    for n in ns:
        ms = sorted(e0.elapsed_time(e1) for e0, e1 in times[n])
        med = ms[len(ms) // 2]
        res[f"n{n}"] = dict(us_per_step_median=1e3 * med / T, us_per_step_min=1e3 * ms[0] / T, us_per_step_max=1e3 * ms[-1] / T,
                            kernels_per_call=kernels[n], kernels_per_step=kernels[n] / T)
    res["overhead_pct"] = 100.0 * (res["n4"]["us_per_step_median"] / res["n0"]["us_per_step_median"] - 1.0)
    print(f"{name}, power limit {power}; B={B} K={K} history {a.hist} tokens, {a.iters} alternating calls per n")
    for n in ns:
        r = res[f"n{n}"]
        print(f"  n={n}: {r['us_per_step_median']:.1f} us/step (median; min {r['us_per_step_min']:.1f}, max {r['us_per_step_max']:.1f}), "
              f"{r['kernels_per_call']} kernels per call = {r['kernels_per_step']:.2f} per step")
    print(f"  n=4 vs n=0: {res['overhead_pct']:+.2f} %")
    print(json.dumps(res))
    if a.json:
        with open(a.json, "w") as f:
            json.dump(res, f, indent=1)
    eng.close()


if __name__ == "__main__":
    main()
