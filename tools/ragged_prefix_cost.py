"""Cost of decoder prefixes of different lengths in one call (a negative id ends an image's prefix, include/gstvd.h gstvd_generate), at
the full config in bf16 with B = 64 images and 150-token synthetic histories (tools/beam_ngram_cost.py:histories), beam-5 and top-k 7
sampling with 4-gram blocking.

    python tools/ragged_prefix_cost.py [--iters 10] [--json out.json] [--parent-lib path/to/parent/libgstvd.so]

Per mode, with CUDA events, medians over alternating rounds (every case once per round):
  * decode step and prefill of a generate call (the method of tools/prefix_cost.py): per-step = (call(T = 18) - call(T = 1)) / 17,
    prefill = call(T = 1) - call(P = 1, T = 1), for uniform P = 1, uniform P = 25 and the ragged batch (lengths drawn from 1..25,
    stride P = 25);
  * a whole round (encoder, cross-K/V prefill, prefix prefill, 18 steps: gstvd_round) of the ragged batch against the same images
    split into one round per distinct length, which is what a caller without ragged prefixes runs.  The split needs one graph per
    length; the lengths are drawn so that they and the ragged round fit the engine's graph pool together (at most 23 lengths).
  * --parent-lib: the decode step of a NULL-prefix call on an engine built from another libgstvd.so (the parent commit's build)
    against this build, alternating in the same process - the per-image length pointer is null there and must cost nothing.
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
from gst_visdial_b200 import _lib  # noqa: E402
from gst_visdial_b200 import weights as W  # noqa: E402
from gst_visdial_b200.engine import Engine  # noqa: E402

P_MAX = 25
MODES = {"beam5": dict(num_beams=5), "sample": dict(num_beams=1, temperature=0.7, top_k=7, top_p=0.0, seed=1, ngram_blocking_size=4)}


def timed(cases, iters):
    """{name: median ms} of the callables in `cases`, every one called once per round, in order."""
    ev = {k: [] for k in cases}
    for _ in range(iters):
        for k, fn in cases.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record()
            ev[k].append((e0, e1))
    torch.cuda.synchronize()
    return {k: sorted(e0.elapsed_time(e1) for e0, e1 in v)[iters // 2] for k, v in ev.items()}


def warm(cases):
    for fn in cases.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()


def make_engine(enc_cfg, dec_cfg, sd, B, lib_path=None, abi=None):
    """An engine on this build, or on the library at lib_path (ABI version abi) when given."""
    if lib_path is None:
        e = Engine(enc_cfg, dec_cfg, dtype="bf16", max_batch=B, max_beams=5)
    else:
        saved = (_lib._lib, _lib.LIB_PATH, _lib.GSTVD_ABI_VERSION)
        _lib._lib, _lib.LIB_PATH, _lib.GSTVD_ABI_VERSION = None, lib_path, abi
        try:
            e = Engine(enc_cfg, dec_cfg, dtype="bf16", max_batch=B, max_beams=5)
        finally:
            _lib._lib, _lib.LIB_PATH, _lib.GSTVD_ABI_VERSION = saved
    e.load_state_dict(sd)
    return e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--hist", type=int, default=150)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--json", default="", help="also write the result here")
    ap.add_argument("--parent-lib", default="", help="libgstvd.so of the parent commit: NULL-prefix decode step, alternating")
    ap.add_argument("--parent-abi", type=int, default=4)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    enc_cfg, dec_cfg = W.load_json_config(W.DEFAULT_ENC_CONFIG), W.load_json_config(W.DEFAULT_DEC_CONFIG)
    B, T = a.batch, 18
    sd = W.synthetic_state_dict(enc_cfg, dec_cfg, seed=0)
    eng = make_engine(enc_cfg, dec_cfg, sd, B)
    b = {k: v.cuda() for k, v in histories(B, a.hist, enc_cfg.vocab_size, enc_cfg.v_feature_size).items()}
    inputs = (b["enc_input_ids"], b["enc_image_feat"], b["enc_image_loc"], b["enc_segments"], b["enc_att_mask"], b["enc_image_mask"])
    out = eng.encode(*inputs)
    eng.prefill_cross(B, out["Le"])
    g = torch.Generator().manual_seed(0)
    base = torch.randint(1000, enc_cfg.vocab_size, (B, P_MAX), generator=g)
    base[:, 0] = 101
    lens = torch.randint(1, P_MAX + 1, (B,), generator=g)
    groups = {int(n): (lens == n).nonzero().flatten().cuda() for n in lens.unique()}
    assert len(groups) <= 23, "the split rounds and the ragged round must fit the graph pool"
    ragged = base.clone()
    for i, n in enumerate(lens.tolist()):
        ragged[i, n:] = -1
    prefixes = {"uniform_P1": base[:, :1].contiguous().cuda(), "uniform_P25": base.cuda(), "ragged": ragged.cuda()}
    hist = dict(hist_ids=b["enc_input_ids"], hist_segments=b["enc_segments"])
    name, power = gpu_info()
    res = dict(gpu=name, power_limit=power, batch=B, hist_tokens=a.hist, new_tokens=T, iters=a.iters, modes=MODES,
               lengths=lens.tolist(), distinct_lengths=len(groups), cases={})
    print(f"{name}, power limit {power}; B={B}, history {a.hist} tokens, lengths 1..{P_MAX} ({len(groups)} distinct), "
          f"{a.iters} alternating rounds, medians")
    for m, mk in MODES.items():
        # decode step and prefill of generate calls, on the cross K/V of all B images (the split rounds leave a subset resident)
        eng.prefill_cross(B, eng.encode(*inputs)["Le"])

        def gen(pre, steps, m=m):
            return lambda: eng.generate(B, max_new_tokens=steps, prefix=prefixes[pre], **hist, **MODES[m])
        cases = {(p, s): gen(p, s) for p in prefixes for s in (T, 1)}
        warm(cases)
        kernels = {}
        for p in prefixes:
            l0 = eng.launch_count
            cases[(p, T)]()
            kernels[p] = eng.launch_count - l0
        med = timed(cases, a.iters)
        for p in prefixes:
            full, one = med[(p, T)], med[(p, 1)]
            r = dict(call_ms=full, call_t1_ms=one, us_per_step=1e3 * (full - one) / (T - 1), prefill_us=1e3 * (one - med[("uniform_P1", 1)]),
                     kernels_per_call=kernels[p])
            res["cases"][f"{m}_{p}"] = r
            print(f"  {m:6s} {p:12s}: call {full:7.3f} ms, {r['us_per_step']:6.1f} us/step, prefill {r['prefill_us']:6.1f} us, "
                  f"{kernels[p]} kernels per call")
        # whole rounds: ragged against one round per length
        def rnd_ragged(m=m):
            return eng.round(*inputs, prefix=prefixes["ragged"], **MODES[m])

        # the per-length inputs are gathered once, outside the timed region
        staged = {n: (tuple(t.index_select(0, idx).contiguous() for t in inputs), base[:, :n].cuda().index_select(0, idx).contiguous())
                  for n, idx in groups.items()}

        def rnd_split(m=m):
            for ins, pre in staged.values():
                eng.round(*ins, prefix=pre, **MODES[m])
        rcases = {"round_ragged": rnd_ragged, "round_split": rnd_split}
        warm(rcases)
        rmed = timed(rcases, a.iters)
        r = dict(round_ragged_ms=rmed["round_ragged"], round_split_ms=rmed["round_split"], split_calls=len(groups))
        res["cases"][f"{m}_rounds"] = r
        print(f"  {m:6s} whole round: ragged {r['round_ragged_ms']:7.3f} ms, split into {len(groups)} per-length rounds "
              f"{r['round_split_ms']:7.3f} ms")
    if a.parent_lib:
        old = make_engine(enc_cfg, dec_cfg, sd, B, a.parent_lib, a.parent_abi)
        for e in (eng, old):
            o = e.encode(*inputs)
            e.prefill_cross(B, o["Le"])
        for m, mk in MODES.items():
            cases = {(who, s): (lambda e=e, s=s, m=m: e.generate(B, max_new_tokens=s, **hist, **MODES[m]))
                     for who, e in (("parent", old), ("this", eng)) for s in (T, 1)}
            warm(cases)
            med = timed(cases, 2 * a.iters)
            r = {who: 1e3 * (med[(who, T)] - med[(who, 1)]) / (T - 1) for who in ("parent", "this")}
            res["cases"][f"{m}_null_prefix_step_us"] = r
            print(f"  {m:6s} NULL prefix decode step: parent build {r['parent']:6.1f} us, this build {r['this']:6.1f} us "
                  f"({100 * (r['this'] / r['parent'] - 1):+.2f} %)")
        old.close()
    print(json.dumps(res))
    if a.json:
        with open(a.json, "w") as f:
            json.dump(res, f, indent=1)
    eng.close()


if __name__ == "__main__":
    main()
