"""Phase timestamps of the deferred-LayerNorm GEMM epilogues next to the plain GEMM (GSTVD_GEMM_TIMES=1)."""
import os
import sys

os.environ.setdefault("GSTVD_GEMM_TIMES", "1")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from gst_visdial_b200 import weights as W  # noqa: E402
from gst_visdial_b200.engine import Engine  # noqa: E402

enc_cfg, dec_cfg = W.load_json_config(W.TINY_ENC_CONFIG), W.load_json_config(W.TINY_DEC_CONFIG)
eng = Engine(enc_cfg, dec_cfg, dtype="bf16", max_batch=4)
M, N = 320, 768
for K1 in (768, 3072):
    a1 = torch.randn(M, K1, device="cuda"); w1 = torch.randn(N, K1, device="cuda") * 0.03; b1 = torch.randn(N, device="cuda")
    res0 = torch.randn(M, N, device="cuda"); g1 = torch.ones(N, device="cuda"); be1 = torch.zeros(N, device="cuda")
    w2 = torch.randn(N, N, device="cuda") * 0.03; b2 = torch.randn(N, device="cuda")
    for rep in range(3):
        sys.stderr.write(f"--- chain M={M} N={N} K1={K1} rep {rep}\n"); sys.stderr.flush()
        eng.op_deferred_ln_chain(a1, w1, b1, res0, g1, be1, w2, b2, g1, be1)
    for rep in range(3):
        sys.stderr.write(f"--- plain M={M} N={N} K={K1} rep {rep}\n"); sys.stderr.flush()
        eng.op_linear(a1, w1, b1, out_dtype="bf16")
eng.close()
