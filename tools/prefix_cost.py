"""Cost of decoding from a decoder prefix: graph replays of the generate call for prefix lengths P in {1, 2, 9, 15, 25}, beam-5
(no blocking, the teacher's setting) and top-k 7 sampling with 4-gram blocking (the questioner's), all cases alternating in one
process, at the full config in bf16 with B = 64 images and 150-token synthetic histories (tools/beam_ngram_cost.py:histories).

    python tools/prefix_cost.py [--iters 20] [--json out.json]

Every case is timed twice per round with CUDA events, as a call of T = 18 new tokens and as a call of T = 1:
  * per-step time  = (call(P, 18) - call(P, 1)) / 17: the mean decode step of a call whose cache holds P - 1 + 18 positions.  Calls
    with P <= 15 hold at most 32 positions and run today's decode kernels; P = 25 holds 42 and runs the 64-position variants;
  * prefill time   = call(P, 1) - call(1, 1): the teacher-forced pass over the first P - 1 prefix positions (its K / V stores
    included) plus the difference of one step at position P - 1 instead of 0 and the copies of the prefix into the context.
Medians over the rounds.  The GPU name and power limit are read in the same run and printed with the numbers.
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

PREFIX_LENS = (1, 2, 9, 15, 25)
MODES = {"beam5": dict(num_beams=5), "sample": dict(num_beams=1, temperature=0.7, top_k=7, top_p=0.0, seed=1, ngram_blocking_size=4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--hist", type=int, default=150)
    ap.add_argument("--iters", type=int, default=20, help="timed rounds; every round calls each case once with T = 18 and once with T = 1")
    ap.add_argument("--json", default="", help="also write the result here")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    enc_cfg, dec_cfg = W.load_json_config(W.DEFAULT_ENC_CONFIG), W.load_json_config(W.DEFAULT_DEC_CONFIG)
    B, T = a.batch, 18
    eng = Engine(enc_cfg, dec_cfg, dtype="bf16", max_batch=B, max_beams=5)
    eng.load_state_dict(W.synthetic_state_dict(enc_cfg, dec_cfg, seed=0))
    b = {k: v.cuda() for k, v in histories(B, a.hist, enc_cfg.vocab_size, enc_cfg.v_feature_size).items()}
    out = eng.encode(b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"], b["enc_image_mask"])
    eng.prefill_cross(B, out["Le"])
    g = torch.Generator().manual_seed(0)
    prefixes = {}
    for P in PREFIX_LENS:
        p = torch.randint(1000, enc_cfg.vocab_size, (B, P), generator=g)
        p[:, 0] = 101
        prefixes[P] = p.cuda()

    def call(mode, P, steps):
        return eng.generate(B, max_new_tokens=steps, prefix=prefixes[P], hist_ids=b["enc_input_ids"], hist_segments=b["enc_segments"],
                            **MODES[mode])

    cases = [(m, P, steps) for m in MODES for P in PREFIX_LENS for steps in (T, 1)]
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
        for P in PREFIX_LENS:
            full, one = med[(m, P, T)], med[(m, P, 1)]
            r = dict(P=P, cached_positions=P - 1 + T, call_ms=full, call_t1_ms=one, us_per_step=1e3 * (full - one) / (T - 1),
                     prefill_us=1e3 * (one - med[(m, 1, 1)]), kernels_per_call=kernels[(m, P, T)])
            res["cases"][f"{m}_P{P}"] = r
            print(f"  {m:6s} P={P:2d} ({r['cached_positions']} positions): call {full:7.3f} ms, {r['us_per_step']:6.1f} us/step, "
                  f"prefill {r['prefill_us']:6.1f} us, {r['kernels_per_call']} kernels per call")
    print(json.dumps(res))
    if a.json:
        with open(a.json, "w") as f:
            json.dump(res, f, indent=1)
    eng.close()


if __name__ == "__main__":
    main()
