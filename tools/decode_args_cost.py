"""Cost of length_penalty, early_stopping and bad_words_ids (include/gstvd.h gstvd_generate): graph replays of the 18-step generate call at
the full config in bf16 with B = 64 images and 150-token synthetic histories (tools/beam_ngram_cost.histories), every case alternating in
one process.

    python tools/decode_args_cost.py [--iters 30] [--json out.json] [--txt out.txt] [--parent-lib path/to/parent/libgstvd.so]

Cases: beam-5 with everything off, with length_penalty 1.5, with early_stopping, with a realistic bad-word list (50 single ids and 50
phrases of two or three ids) and with a list at the caps (1024 sequences, 4096 ids); top-k 7 sampling (temperature 0.7, 4-gram question
blocking, as the questioner runs) without and with the realistic and the capped list.  Per case: the device time of one generate call
(CUDA events, median over the alternating replays) divided by its 18 decode steps, and the kernels per call (gstvd_launch_count).
--parent-lib: the everything-off beam-5 and sampling steps on an engine built from another libgstvd.so (the parent commit's build),
alternating with this build in the same process.  The GPU name and power limit are read in the same run.
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
from ragged_prefix_cost import make_engine  # noqa: E402
from gst_visdial_b200 import weights as W  # noqa: E402

BEAM = dict(num_beams=5)
SAMPLE = dict(temperature=0.7, top_k=7, top_p=0.0, seed=1, ngram_blocking_size=4)


def word_lists(vocab):
    """(realistic, capped) bad-word lists drawn from a seeded generator over ordinary ids (1000 .. vocab)."""
    g = torch.Generator().manual_seed(0)
    ids = lambda n: torch.randint(1000, vocab, (n,), generator=g).tolist()    # noqa: E731
    realistic = [[w] for w in ids(50)] + [ids(2 + i % 2) for i in range(50)]
    capped = [[w] for w in ids(256)] + [ids(5) for _ in range(768)]          # 1024 sequences, 256 + 768 * 5 = 4096 ids
    assert len(capped) == 1024 and sum(map(len, capped)) == 4096
    return realistic, capped


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--hist", type=int, default=150)
    ap.add_argument("--iters", type=int, default=30, help="timed calls per case (alternating)")
    ap.add_argument("--json", default="", help="also write the result here")
    ap.add_argument("--txt", default="", help="also write the printed summary here")
    ap.add_argument("--parent-lib", default="", help="libgstvd.so of the parent commit: everything-off decode steps, alternating")
    ap.add_argument("--parent-abi", type=int, default=6)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    enc_cfg, dec_cfg = W.load_json_config(W.DEFAULT_ENC_CONFIG), W.load_json_config(W.DEFAULT_DEC_CONFIG)
    B, T = a.batch, 18
    sd = W.synthetic_state_dict(enc_cfg, dec_cfg, seed=0)
    engines = {"this": make_engine(enc_cfg, dec_cfg, sd, B)}
    if a.parent_lib:
        engines["parent"] = make_engine(enc_cfg, dec_cfg, sd, B, a.parent_lib, a.parent_abi)
    b = {k: v.cuda() for k, v in histories(B, a.hist, enc_cfg.vocab_size, enc_cfg.v_feature_size).items()}
    rnd = (b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"], b["enc_image_mask"])
    hist = dict(hist_ids=b["enc_input_ids"], hist_segments=b["enc_segments"])
    for e in engines.values():
        e.round(*rnd, num_beams=5)                                 # leaves the cross-K/V of the B images resident
    realistic, capped = word_lists(enc_cfg.vocab_size)
    cases = {"beam5_off": ("this", BEAM), "beam5_length_penalty_1.5": ("this", dict(BEAM, length_penalty=1.5)),
             "beam5_early_stopping": ("this", dict(BEAM, early_stopping=True)),
             "beam5_bad_words_realistic": ("this", dict(BEAM, bad_words_ids=realistic)),
             "beam5_bad_words_caps": ("this", dict(BEAM, bad_words_ids=capped)),
             "sample_topk7_off": ("this", SAMPLE), "sample_topk7_bad_words_realistic": ("this", dict(SAMPLE, bad_words_ids=realistic)),
             "sample_topk7_bad_words_caps": ("this", dict(SAMPLE, bad_words_ids=capped))}
    if a.parent_lib:
        cases.update({"beam5_off_parent_build": ("parent", BEAM), "sample_topk7_off_parent_build": ("parent", SAMPLE)})

    def call(c):
        who, kw = cases[c]
        engines[who].generate(B, **hist, **kw)

    kernels = {}
    for c in cases:                                                # capture + warm up every graph
        for _ in range(3):
            call(c)
        torch.cuda.synchronize()
        before = engines[cases[c][0]].launch_count
        call(c)
        kernels[c] = engines[cases[c][0]].launch_count - before
    times = {c: [] for c in cases}
    for _ in range(a.iters):
        for c in cases:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); call(c); e1.record()
            times[c].append((e0, e1))
    torch.cuda.synchronize()
    name, power = gpu_info()
    res = dict(gpu=name, power_limit=power, batch=B, hist_tokens=a.hist, steps=T, iters=a.iters, realistic_list=dict(
        single=50, phrases=50, ids=sum(map(len, realistic))), capped_list=dict(sequences=len(capped), ids=sum(map(len, capped))), cases={})
    lines = [f"{name}, power limit {power}; full config bf16, B={B}, history {a.hist} tokens, {a.iters} alternating graph replays per case"]
    ms = {c: sorted(e0.elapsed_time(e1) for e0, e1 in times[c]) for c in cases}
    for c in cases:
        m = ms[c]
        med = m[len(m) // 2]
        base = ms["beam5_off" if c.startswith("beam5") else "sample_topk7_off"][len(m) // 2]
        r = dict(us_per_step_median=1e3 * med / T, us_per_step_min=1e3 * m[0] / T, us_per_step_max=1e3 * m[-1] / T,
                 kernels_per_call=kernels[c], vs_off_pct=100.0 * (med / base - 1.0))
        res["cases"][c] = r
        lines.append(f"  {c}: {r['us_per_step_median']:.1f} us/step (median; min {r['us_per_step_min']:.1f}, max {r['us_per_step_max']:.1f}), "
                     f"{r['kernels_per_call']} kernels per call, {r['vs_off_pct']:+.2f} % vs off on this build")
    text = "\n".join(lines)
    print(text)
    print(json.dumps(res))
    if a.json:
        with open(a.json, "w") as f:
            json.dump(res, f, indent=1)
    if a.txt:
        with open(a.txt, "w") as f:
            f.write(text + "\n")
    for e in engines.values():
        e.close()


if __name__ == "__main__":
    main()
