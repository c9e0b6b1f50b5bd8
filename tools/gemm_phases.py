"""Phase timestamps of the tcgen05 GEMM on the decode-step shapes (GSTVD_GEMM_TIMES=1 makes gstvd_op_linear print them)."""
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
M = int(sys.argv[1]) if len(sys.argv) > 1 else 320
for N, K in ((768, 768), (2304, 768), (3072, 768), (768, 3072), (30522, 768)):
    a = torch.randn(M, K, device="cuda")
    w = torch.randn(N, K, device="cuda") * 0.03
    b = torch.randn(N, device="cuda")
    for rep in range(3):
        sys.stderr.write(f"--- M={M} N={N} K={K} rep {rep}\n"); sys.stderr.flush()
        eng.op_linear(a, w, b, out_dtype="bf16")
eng.close()
