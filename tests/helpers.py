"""Shared test helpers (test infrastructure: may import oracle/)."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from gst_visdial_b200 import synthetic as S  # noqa: E402
from oracle import restatement as R  # noqa: E402


def history_batch(enc_cfg, start, count, rounds=2):
    """Same construction as oracle/gen_golden.py:history_batch (kept in sync by test_oracle_golden)."""
    b = S.synthetic_batch(start, count, vocab_size=enc_cfg.vocab_size, v_feature_size=enc_cfg.v_feature_size)
    ids, seg = b["enc_input_ids"], b["enc_segments"]
    enc_len = (ids != 0).sum(-1)
    abnormal = set()
    for r in range(rounds):
        q = torch.stack([S.synthetic_utterance(start + i, 2 * r, enc_cfg.vocab_size) for i in range(count)])
        enc_len += R.splice(ids, seg, enc_len, q, None, abnormal)
        a = torch.stack([S.synthetic_utterance(start + i, 2 * r + 1, enc_cfg.vocab_size) for i in range(count)])
        a = a.masked_fill(a == R.EOS, 0)
        enc_len += R.splice(ids, seg, enc_len, a, 1, abnormal)
    b["enc_att_mask"] = (ids != 0).float()
    return b


def load_golden(golden_dir, tag):
    """Arrays of <tag>.npz and of its continuation files <tag>.part2.npz, ... (oracle/gen_golden.py:save_golden)."""
    g = dict(np.load(os.path.join(golden_dir, f"{tag}.npz")))
    i = 2
    while os.path.exists(os.path.join(golden_dir, f"{tag}.part{i}.npz")):
        g.update(np.load(os.path.join(golden_dir, f"{tag}.part{i}.npz")))
        i += 1
    return g


def rel_rms(a: torch.Tensor, ref: torch.Tensor) -> float:
    return float((a.double() - ref.double()).pow(2).mean().sqrt() / ref.double().pow(2).mean().sqrt().clamp(min=1e-30))


def max_abs(a: torch.Tensor, ref: torch.Tensor) -> float:
    return float((a.double() - ref.double()).abs().max())


def bf16_report(a: torch.Tensor, ref: torch.Tensor, rtol: float = 2e-2) -> dict:
    """The three readings of "2e-2 relative" (SURVEY.md 8d) for rows [n, width]: rel-rms over everything; the worst
    max|delta| / rms(reference row); and the share of elements with |delta| <= rtol * rms(row) + rtol * |ref| (the elementwise
    rtol = atol/rms = 2e-2 pass rate)."""
    a, ref = a.double().reshape(-1, a.shape[-1]), ref.double().reshape(-1, ref.shape[-1])
    d = (a - ref).abs()
    row_rms = ref.pow(2).mean(-1, keepdim=True).sqrt().clamp(min=1e-30)
    return {
        "rel_rms": float((a - ref).pow(2).mean().sqrt() / ref.pow(2).mean().sqrt().clamp(min=1e-30)),
        "max_over_row_rms": float((d.max(-1, keepdim=True).values / row_rms).max()),
        "pass_rate": float((d <= rtol * row_rms + rtol * ref.abs()).double().mean()),
        "max_abs": float(d.max()),
    }
