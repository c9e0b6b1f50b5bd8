"""GPU: every tcgen05 GEMM variant and epilogue the engine launches, forced one at a time, against an fp64 reference.

The variants run through the single-operator entries of the C ABI (gstvd_op_linear, gstvd_op_linear_ln) with the kernel and store
forced (include/gstvd.h lists what each kernel can run); each entry reports the (kernel, store) it launched.  The reference is fp64
on the same bf16-rounded operands, computed on the GPU.  Every element is checked against a bound written down here, not fitted to a
run (u = 2^-24, the fp32 unit roundoff):
  accumulation   K u (|A| |W|^T)    fp32 accumulation of K products, plus u |y| for the bias add;
  GELU           the fast GELU of the tcgen05 epilogues errs by <= 2.5e-4 |x| and < 2e-4 (gemm_tc.cuh, gelu_fast), and passes the
                 accumulation error on with a slope of at most 1.13;
  bf16 output    one bf16 ulp of the result.
The worst error / bound ratio of every case is printed ("[gemm] ..." lines, pytest -s).

Exactness checks catch a misplaced element that a tolerance would hide: every tcgen05 variant of one problem and output type gives
identical bits (same products, same k order, fp32 accumulation in the tensor core; only the SIMT kernel sums differently); each
variant's bf16 output is its fp32 output rounded to bf16; the output buffer starts as NaN, so columns N .. ldc-1 must still be NaN
and, head-major, no element may be.
"""
import math

import pytest
import torch

from gst_visdial_b200._lib import GEMM_KERNELS, GEMM_STORES, GstvdError

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
GELU_SLOPE = 1.13                      # max |GELU'(x)| = 1.1289 (at x = sqrt 2)
UNSUPPORTED = -3
TC = ("tc32", "tc64", "tc128", "tc256")
CHUNKED = ("tc32", "tc64", "skinny32", "skinny64", "ln32", "ln64")      # whole 64-element k-chunks: K % 64 == 0
WORST = {}                             # variant -> worst error / bound over the file


@pytest.fixture(scope="module")
def eng(full_cfgs):
    from gst_visdial_b200.engine import Engine
    enc_cfg, dec_cfg = full_cfgs
    e = Engine(enc_cfg, dec_cfg, device=0, dtype="bf16", max_batch=8, max_beams=5)
    yield e
    e.close()
    if WORST:
        print("\n[gemm] worst error / bound per variant: " + ", ".join(f"{k} {v:.3f}" for k, v in sorted(WORST.items())))


def bf16(t):
    return t.bfloat16().float()


def ulp_bf16(x):
    """One bf16 ulp of |x| (fp64): 2^(floor(log2 |x|) - 7)."""
    _, e = torch.frexp(x.abs().float())
    return torch.ldexp(torch.ones_like(x), (e - 8).to(x.device)).double()


def gelu64(x):
    return x * 0.5 * (1.0 + torch.erf(x / math.sqrt(2.0)))


def ref_linear(a, w, b, act, out_bf16, simt=False):
    """fp64 reference and bound of act(a w^T + b) on the GPU for bf16-rounded fp32 operands a [M, K], w [N, K]."""
    a64, w64 = a.cuda().double(), w.cuda().double()
    y = a64 @ w64.t()
    K = a.shape[1]
    if a.shape[0] * w.shape[0] * K <= 2e10:
        mag = a64.abs() @ w64.abs().t()
    else:                                   # looser, cheaper: |A| |W|^T <= rowsum |A| x max |W_n|
        mag = a64.abs().sum(1, keepdim=True) * w64.abs().amax(1)[None, :]
    bound = K * U * mag
    if b is not None:
        y = y + b.cuda().double()
    bound = bound + U * y.abs()
    if act:
        x = y
        y = gelu64(x)
        g_err = (1e-7 * x.abs()).clamp(max=1e-7) if simt else (2.5e-4 * x.abs()).clamp(max=2e-4)
        bound = GELU_SLOPE * bound + g_err
    if out_bf16:
        bound = bound + ulp_bf16(y.abs() + bound)
    return y, bound


def worst_ratio(y, ref, bound, what, variant):
    err = (y.double() - ref).abs()
    ratio = float((err / bound).max())
    print(f"[gemm] {what}: worst error / bound {ratio:.3f}")
    WORST[variant] = max(WORST.get(variant, 0.0), ratio)
    return ratio


def operands(M, N, K, seed, bias=True):
    g = torch.Generator().manual_seed(seed)
    a = bf16(torch.randn(M, K, generator=g))
    w = bf16(torch.randn(N, K, generator=g) / math.sqrt(K))
    b = torch.randn(N, generator=g) if bias else None
    return a.cuda(), w.cuda(), None if b is None else b.cuda()


# ---- what each kernel can run (include/gstvd.h); the launcher must refuse everything else ----------------------------------------
def can_run(kernel, store, out_f32, K, ldc_bytes_ok, hm=None, M=None):
    if kernel == "simt":
        return store == "generic"
    if K % 8 or (kernel in CHUNKED and K % 64):
        return False
    if kernel.startswith("skinny"):
        return store == "direct" and hm is None and ldc_bytes_ok
    if kernel.startswith("pair") and store != "tma":
        return False
    if store == "tma":
        if hm is not None:
            return kernel in ("tc128", "tc256", "pair128", "pair256") and not out_f32 and M == hm[3] * hm[1]
        return ldc_bytes_ok
    if store == "direct":
        return hm is None and ldc_bytes_ok
    return kernel in TC


PLAIN_VARIANTS = [(k, s) for k in TC for s in ("generic", "tma", "direct")] + [("skinny32", "direct"), ("skinny64", "direct"),
                                                                                ("pair128", "tma"), ("pair256", "tma"), ("simt", "generic")]

# Plain epilogues.  Between them every variant sees a partial last row tile (of 128 rows, 64 rows skinny, a half-empty pair tile),
# a partial last 32-column block (N = 40, 3000, 30522), at least three tiles per resident CTA so the two TMEM accumulator stages wrap
# (M = 4700, N = 3000: 37 x 12 tiles of 128 x 256 over 148 CTAs, 19 x 12 pair tiles over 74 pairs, 74 x 94 skinny tiles over 296),
# K % 64 != 0 (K = 72, where the kernel allows it), bias / no bias, GELU.  (M, N, K, ldc, act, bias)
PLAIN_CASES = [
    (4700, 3000, 768, 3000, 1, True),      # the wrap case, every variant
    (1100, 1000, 72, 1000, 0, False),      # K tail zero-filled by TMA (tc128 / tc256 / pairs / simt)
    (129, 40, 64, 40, 1, True),            # one partial 32-column block
    (65, 96, 768, 96, 0, True),
    (17, 768, 2048, 768, 1, False),
    (1, 768, 768, 768, 0, True),
    (320, 2304, 768, 2304, 0, True),       # decode-step q|k|v
    (513, 3072, 768, 3072, 1, True),       # decode-step FFN1 one past the skinny rule
    (320, 30522, 768, 30528, 0, True),     # LM head: logits rows of Vpad = 30528 (fp32 only)
    (32, 30522, 768, 30528, 0, True),
    (5, 2, 768, 2, 0, True),               # NSP head: 8-byte rows, generic store only
    (129, 40, 64, 41, 0, True),            # odd bf16 row stride (element stores, the ld_even branch)
]


@pytest.mark.parametrize("M,N,K,ldc,act,bias", PLAIN_CASES)
def test_plain_epilogues(eng, M, N, K, ldc, act, bias):
    a, w, b = operands(M, N, K, M * 7 + N * 3 + K, bias)
    outs = ("fp32",) if N > 4000 else ("fp32", "bf16")
    ref = {o: ref_linear(a, w, b, act, o == "bf16") for o in outs}
    ref_simt = ref_linear(a, w, b, act, False, simt=True)
    results = {}
    for out in outs:
        esz = 4 if out == "fp32" else 2
        for kernel, store in PLAIN_VARIANTS:
            if kernel == "simt" and out == "bf16":
                continue
            if not can_run(kernel, store, out == "fp32", K, (ldc * esz) % 16 == 0):
                continue
            y, ran = eng.op_linear(a, w, b, act=act, dtype="bf16", out_dtype=out, ldc=ldc, kernel=kernel, store=store, want_variant=True)
            what = f"{kernel}/{store} {out} M={M} N={N} K={K} ldc={ldc} act={act} bias={bias}"
            assert ran == (kernel, store.lower()), what
            assert bool(y[:, N:].isnan().all()), f"{what}: wrote past column N"
            y = y[:, :N]
            assert not bool(y.isnan().any()), f"{what}: element not written"
            r, bd = ref_simt if kernel == "simt" else ref[out]
            assert worst_ratio(y, r, bd, what, f"{kernel}/{store}/{out}") <= 1.0, what
            results[(kernel, store, out)] = y
    tc_keys = [k for k in results if k[0] != "simt"]
    for out in outs:
        keys = [k for k in tc_keys if k[2] == out]
        for k in keys[1:]:
            assert torch.equal(results[k], results[keys[0]]), f"{k} differs from {keys[0]} in bits (M={M} N={N} K={K})"
    for (kernel, store, out), y in results.items():
        if out == "bf16":
            assert torch.equal(y, bf16(results[(kernel, store, "fp32")])), f"{kernel}/{store}: bf16 output is not the rounded fp32 output"


# ---- head-major scatter (cross-attention K/V prefill) ---------------------------------------------------------------------------
# (D, L, B, layers, heads): G = 2 * heads column groups of D per layer; L either side of the 128-row tiles, L = 1; B = 64 images
HM_CASES = [(64, 293, 3, 1, 12), (32, 37, 64, 1, 2), (128, 129, 1, 6, 6), (64, 128, 3, 6, 12), (64, 1, 64, 1, 12), (32, 127, 3, 1, 2)]
HM_VARIANTS = [(k, "generic") for k in TC] + [("tc128", "tma"), ("tc256", "tma"), ("pair128", "tma"), ("pair256", "tma")]


def hm_layout(y, D, L, B, layers, G):
    """[M = B * L, N = layers * G * D] -> [layers][B][G][L][D]."""
    return y.reshape(B, L, layers, G, D).permute(2, 0, 3, 1, 4)


@pytest.mark.parametrize("D,L,B,layers,heads", HM_CASES)
def test_head_major(eng, D, L, B, layers, heads):
    G = 2 * heads
    M, N, K = B * L, layers * G * D, 768
    a, w, b = operands(M, N, K, D + 7 * L + 31 * B + layers)
    hm = (D, L, G, B)
    r, bd = ref_linear(a, w, b, 0, True)
    r, bd = hm_layout(r, D, L, B, layers, G), hm_layout(bd, D, L, B, layers, G)
    plain = eng.op_linear(a, w, b, dtype="bf16", out_dtype="bf16", kernel="tc128", store="generic")
    plain = hm_layout(plain, D, L, B, layers, G)
    for kernel, store in HM_VARIANTS:
        y, ran = eng.op_linear(a, w, b, dtype="bf16", out_dtype="bf16", hm=hm, kernel=kernel, store=store, want_variant=True)
        what = f"{kernel}/{store} head-major D={D} L={L} B={B} layers={layers} G={G}"
        assert ran == (kernel, store), what
        assert not bool(y.isnan().any()), f"{what}: element not written"
        assert worst_ratio(y, r, bd, what, f"{kernel}/{store}/hm") <= 1.0, what
        assert torch.equal(y, plain), f"{what}: differs from the row-major result scattered on the host"
    for kernel in TC:                                    # fp32 output: generic store only (the TMA store writes bf16)
        y = eng.op_linear(a, w, b, dtype="bf16", out_dtype="fp32", hm=hm, kernel=kernel, store="generic")
        assert not bool(y.isnan().any())
        assert torch.equal(bf16(y), plain), f"{kernel}/generic fp32 head-major"
    y = eng.op_linear(a, w, b, dtype="fp32", out_dtype="fp32", hm=hm, kernel="simt", store="generic")
    r32, bd32 = ref_linear(a, w, b, 0, False, simt=True)
    assert worst_ratio(y, hm_layout(r32, D, L, B, layers, G), hm_layout(bd32, D, L, B, layers, G), f"simt head-major D={D} L={L} B={B}",
                       "simt/generic/hm") <= 1.0


# ---- deferred LayerNorm (decode step) ------------------------------------------------------------------------------------------
LN_COMBOS = {        # name: (fold, act, residual: None / "raw" / "ln", stats_out)
    "fold": (True, 0, None, False),                  # q|k|v of layers 1.. and the cross query
    "fold_gelu": (True, 1, None, False),             # FFN1
    "raw_res_stats": (False, 0, "raw", True),        # attention output
    "ln_res_stats": (False, 0, "ln", True),          # cross-attention output, FFN2
    "fold_ln_res_stats": (True, 0, "ln", True),      # no production call site; the producer -> consumer chain test uses it
}
LN_SHAPES = [(768, 768), (2304, 768), (3072, 768), (768, 3072)]
LN_M = [1, 5, 64, 65, 320, 512]


def ln_valid(combo, N, K):
    fold, _, res, stats = LN_COMBOS[combo]
    return not (fold and K > 1024) and not ((res == "ln" or stats) and N > 1024)


LN_CASES = [(c, N, K) for c in LN_COMBOS for N, K in LN_SHAPES if ln_valid(c, N, K)]


def ln_rows(M, W, g):
    """Rows with a common offset of about 8 and an outlier column of about +-40 (bf16-rounded)."""
    x = torch.randn(M, W, generator=g) + 8.0
    x[:, 5] = 40.0 * torch.where(torch.rand(M, generator=g) < 0.5, -1.0, 1.0)
    return bf16(x)


def part_stats(x):
    """Per-32-column (mean, M2) of rows x [M, W] in the GemmArgs layout [W/32][M][2], fp64 -> fp32."""
    M, W = x.shape
    xb = x.double().reshape(M, W // 32, 32)
    mean = xb.mean(-1)
    m2 = (xb - mean[..., None]).pow(2).sum(-1)
    return torch.stack([mean, m2], -1).permute(1, 0, 2).float().contiguous()


def merged(st):
    """(mean, rstd) fp64 [M] of the partials st [P][M][2], merged as the kernel does (equal counts of 32; eps 1e-12)."""
    st = st.double()
    P = st.shape[0]
    mean = st[..., 0].mean(0)
    m2 = st[..., 1].sum(0) + 32.0 * (st[..., 0] - mean).pow(2).sum(0)
    return mean, 1.0 / torch.sqrt(m2 / (32 * P) + 1e-12)


@pytest.mark.parametrize("kernel", ["ln32", "ln64"])
@pytest.mark.parametrize("M", LN_M)
@pytest.mark.parametrize("combo,N,K", LN_CASES)
def test_deferred_ln_epilogue(eng, kernel, M, combo, N, K):
    fold, act, res_kind, want_stats = LN_COMBOS[combo]
    g = torch.Generator().manual_seed(M * 131 + N * 7 + K + len(combo))
    a = ln_rows(M, K, g) if fold else bf16(torch.randn(M, K, generator=g))
    w = torch.randn(N, K, generator=g) / math.sqrt(K)
    bias = torch.randn(N, generator=g)
    gam, bet = 1.0 + 0.2 * torch.randn(K, generator=g), 0.1 * torch.randn(K, generator=g)
    res = ln_rows(M, N, g) if res_kind else None
    rgam, rbet = 1.0 + 0.2 * torch.randn(N, generator=g), 0.1 * torch.randn(N, generator=g)
    a_st = part_stats(a) if fold else None
    r_st = part_stats(res) if res_kind == "ln" else None
    y, st, ran = eng.op_linear_ln(a, w, bias, a_stats=a_st, ln_gamma=gam if fold else None, ln_beta=bet if fold else None, res=res,
                                  res_stats=r_st, res_gamma=rgam if r_st is not None else None, res_beta=rbet if r_st is not None else None,
                                  act=act, want_stats=want_stats, kernel=kernel)
    what = f"{kernel} {combo} M={M} N={N} K={K}"
    assert ran == (kernel, "direct"), what
    a64, w64, b64 = a.cuda().double(), w.cuda().double(), bias.cuda().double()
    if fold:
        # the kernel's arithmetic in fp64: W' = bf16(fp32(W gamma)), c = sum_k W', d = sum_k beta_k W_nk + b, rstd (A W'^T - mean c) + d
        wf = bf16(w * gam[None, :]).cuda().double()
        c = wf.sum(1)
        d = w64 @ bet.cuda().double() + b64
        mean, rstd = merged(a_st.cuda())
        acc = a64 @ wf.t()
        pre = rstd[:, None] * (acc - mean[:, None] * c[None, :]) + d[None, :]
        # accumulation of A W'^T and of c (K products each); the fp32 merge of the P = K / 32 partial statistics ((2P + 8) u relative
        # on mean and rstd); the fp32 sum of d; the fp32 operations of the epilogue
        P = K // 32
        mmax = a_st[..., 0].cuda().double().abs().amax(0)
        centred = (acc - mean[:, None] * c[None, :]).abs()
        bound = (rstd[:, None] * (K * U * (a64.abs() @ wf.abs().t()) + K * U * mmax[:, None] * wf.abs().sum(1)[None, :]
                                  + (2 * P + 8) * U * (centred + mmax[:, None] * c.abs()[None, :]))
                 + K * U * (w64.abs() @ bet.cuda().double().abs())[None, :] + 4 * U * (pre.abs() + d.abs()[None, :]))
        # plain LN-then-linear: differs by the rounding of W gamma to bf16 (2^-9 relative per weight)
        xhat = (a64 - mean[:, None]) * rstd[:, None]
        plain = (xhat * gam.cuda().double() + bet.cuda().double()) @ w64.t() + b64
        plain_extra = 2.0 ** -9 * (xhat.abs() @ (w64 * gam.cuda().double()).abs().t())
    else:
        w16 = bf16(w).cuda().double()
        pre = a64 @ w16.t() + b64
        bound = K * U * (a64.abs() @ w16.abs().t()) + U * pre.abs()
        plain, plain_extra = pre, torch.zeros_like(pre)
    if res_kind:
        r64 = res.cuda().double()
        if res_kind == "ln":
            rmean, rrstd = merged(r_st.cuda())
            rn = (r64 - rmean[:, None]) * rrstd[:, None]
            r64 = rn * rgam.cuda().double() + rbet.cuda().double()
            Pr = N // 32
            rmax = r_st[..., 0].cuda().double().abs().amax(0)
            bound = bound + ((2 * Pr + 8) * U * (rn.abs() + rmax[:, None] * rrstd[:, None]) * rgam.cuda().double().abs()
                             + 2 * U * rbet.cuda().double().abs())
        pre, plain = pre + r64, plain + r64
        bound = bound + U * pre.abs()
    if act:
        bound = GELU_SLOPE * bound + (2.5e-4 * pre.abs()).clamp(max=2e-4)
        pre, plain = gelu64(pre), gelu64(plain)
        plain_extra = GELU_SLOPE * plain_extra
    bound = bound + ulp_bf16(pre.abs() + bound)
    assert not bool(y.isnan().any()), what
    assert worst_ratio(y, pre, bound, what, f"{kernel}/{combo}") <= 1.0, what
    assert float(((y.double() - plain).abs() / (bound + plain_extra)).max()) <= 1.0, f"{what}: far from LayerNorm-then-linear"
    if want_stats:
        yb = y.double().reshape(M, N // 32, 32)
        shift = yb[..., 0]
        mean_ref = yb.mean(-1)
        m2_ref = (yb - mean_ref[..., None]).pow(2).sum(-1)
        dev = (yb - shift[..., None]).abs()
        st = st.double().permute(1, 0, 2)
        mean_bd = 64 * U * (shift.abs() + dev.mean(-1)) + 1e-300
        m2_bd = 128 * U * dev.pow(2).sum(-1) + 1e-300
        assert bool(((st[..., 0] - mean_ref).abs() <= mean_bd).all()), f"{what}: stats_out mean"
        assert bool(((st[..., 1] - m2_ref).abs() <= m2_bd).all()), f"{what}: stats_out M2"


# ---- production shapes, the engine's own choice ---------------------------------------------------------------------------------
def production_shapes(full_cfgs):
    """(label, M, N, K, ldc, act, out_dtype, hm) of the engine's GEMM call sites (csrc/engine.cu) at the benchmark batches."""
    enc, dec = full_cfgs
    H, F, Hv, Fv, Hb, Vf = enc.hidden_size, enc.intermediate_size, enc.v_hidden_size, enc.v_intermediate_size, enc.bi_hidden_size, enc.v_feature_size
    V = dec.vocab_size
    Vpad = (V + 7) // 8 * 8
    Lt, Lv = 256, 37
    heads = dec.num_attention_heads
    shapes = []
    for B in (32, 64):                                   # gen_qa_ppl / gen_teacher batches (bench.py)
        Mt, Mv = B * Lt, B * Lv
        shapes += [(f"text qkv B={B}", Mt, 3 * H, H), (f"text out B={B}", Mt, H, H), (f"text ffn1 B={B}", Mt, F, H, 1),
                   (f"text ffn2 B={B}", Mt, H, F), (f"image embed B={B}", Mv, Hv, Vf), (f"image qkv B={B}", Mv, 3 * Hv, Hv),
                   (f"image ffn1 B={B}", Mv, Fv, Hv, 1), (f"co-attn qkv1 B={B}", Mv, 3 * Hb, Hv), (f"co-attn qkv2 B={B}", Mt, 3 * Hb, H),
                   (f"fusion fc_v B={B}", Mv, H, Hv)]
    for M in (32, 320):                                  # decode step: 32 sampled rows, 64 images x 5 beams
        shapes += [(f"decode qkv M={M}", M, 3 * H, H), (f"decode out M={M}", M, H, H), (f"decode ffn1 M={M}", M, dec.intermediate_size, H, 1),
                   (f"decode ffn2 M={M}", M, H, dec.intermediate_size),
                   (f"LM head M={M}", M, V, H, 0, Vpad, "fp32")]
    D = H // heads
    shapes.append((f"cross K/V prefill B=8", 8 * (Lv + Lt), dec.num_hidden_layers * 2 * H, H, 0, None, "bf16", (D, Lv + Lt, 2 * heads, 8)))
    out = []
    for s in shapes:
        label, M, N, K = s[:4]
        act = s[4] if len(s) > 4 else 0
        ldc = s[5] if len(s) > 5 else None
        od = s[6] if len(s) > 6 else "bf16"
        hm = s[7] if len(s) > 7 else None
        out.append((label, M, N, K, act, ldc, od, hm))
    return out


def test_production_shapes_auto(eng, full_cfgs):
    """Call sites: engine.cu Exec::gemm from do_encode (text / image / co-attention / fusion layers), decode_step (:754-767, the LM
    head with ldc = Vpad at :767), do_prefill (:592, head-major).  Each runs the engine's own choice, which must be a variant the
    forced tests above cover, and is compared with fp64."""
    covered = set(PLAIN_VARIANTS) | set(HM_VARIANTS)
    for label, M, N, K, act, ldc, od, hm in production_shapes(full_cfgs):
        a, w, b = operands(M, N, K, M + N + K)
        y, ran = eng.op_linear(a, w, b, act=act, dtype="bf16", out_dtype=od, ldc=ldc, hm=hm, want_variant=True)
        print(f"[gemm] production {label}: M={M} N={N} K={K} ran {ran[0]}/{ran[1]}")
        assert ran in covered, f"{label}: {ran} is not in the forced matrix"
        r, bd = ref_linear(a, w, b, act, od == "bf16")
        if hm is not None:
            D, L, G, B = hm
            r, bd = hm_layout(r, D, L, B, N // (D * G), G), hm_layout(bd, D, L, B, N // (D * G), G)
        else:
            assert bool(y[:, N:].isnan().all()), label
            y = y[:, :N]
        assert worst_ratio(y, r, bd, f"production {label} ({ran[0]}/{ran[1]})", f"{ran[0]}/{ran[1]}/{od}") <= 1.0, label
    # the decode step's deferred-LayerNorm GEMMs (engine.cu:734-747) at M = 32 and 320
    H = full_cfgs[1].hidden_size
    F = full_cfgs[1].intermediate_size
    for M in (32, 320):
        g = torch.Generator().manual_seed(M)
        for label, N, K, fold, act, res in (("qkv", 3 * H, H, True, 0, None), ("ffn1", F, H, True, 1, None), ("out", H, H, False, 0, "raw"),
                                            ("ffn2", H, F, False, 0, "ln")):
            a = ln_rows(M, K, g)
            w = torch.randn(N, K, generator=g) / math.sqrt(K)
            r = ln_rows(M, N, g) if res else None
            y, st, ran = eng.op_linear_ln(a, w, torch.randn(N, generator=g), a_stats=part_stats(a) if fold else None,
                                          ln_gamma=torch.ones(K) if fold else None, ln_beta=torch.zeros(K) if fold else None, res=r,
                                          res_stats=part_stats(r) if res == "ln" else None, res_gamma=torch.ones(N) if res == "ln" else None,
                                          res_beta=torch.zeros(N) if res == "ln" else None, act=act, want_stats=res is not None)
            print(f"[gemm] production deferred-LN {label} M={M}: ran {ran[0]}/{ran[1]}")
            assert ran in (("ln32", "direct"), ("ln64", "direct")) and torch.isfinite(y).all(), label


# ---- refusals ------------------------------------------------------------------------------------------------------------------
REFUSED = [  # (kernel, store, M, N, K, ldc, out_dtype, hm)
    ("skinny32", "tma", 64, 96, 768, None, "fp32", None), ("skinny64", "generic", 64, 96, 768, None, "bf16", None),
    ("pair128", "direct", 2048, 256, 768, None, "bf16", None), ("pair256", "generic", 2048, 256, 768, None, "fp32", None),
    ("tc32", "generic", 64, 96, 72, None, "fp32", None), ("skinny32", "direct", 64, 96, 72, None, "fp32", None),
    ("tc128", "tma", 5, 2, 768, 2, "fp32", None), ("tc64", "direct", 5, 41, 768, 41, "bf16", None),
    ("tc32", "tma", 129, 128, 768, None, "bf16", (64, 129, 2, 1)), ("tc128", "direct", 129, 128, 768, None, "bf16", (64, 129, 2, 1)),
    ("tc128", "tma", 129, 128, 768, None, "fp32", (64, 129, 2, 1)), ("skinny32", "direct", 129, 128, 768, None, "bf16", (64, 129, 2, 1)),
    ("ln32", "direct", 64, 96, 768, None, "bf16", None), ("tc128", None, 64, 96, 68, None, "fp32", None),
]


@pytest.mark.parametrize("kernel,store,M,N,K,ldc,od,hm", REFUSED)
def test_refusals(eng, kernel, store, M, N, K, ldc, od, hm):
    """A forced variant that cannot run its arguments is refused with GSTVD_ERR_UNSUPPORTED before anything is launched."""
    a, w, b = operands(M, N, K, 5)
    before = eng.launch_count
    with pytest.raises(GstvdError) as e:
        eng.op_linear(a, w, b, dtype="bf16", out_dtype=od, ldc=ldc, hm=hm, kernel=kernel, store=store)
    assert e.value.status == UNSUPPORTED, str(e.value)
    assert eng.launch_count == before


def test_ln_refusals(eng):
    M, N, K = 64, 768, 768
    a = torch.randn(M, K)
    w = torch.randn(N, K)
    res = torch.randn(M, N)
    before = eng.launch_count
    for kernel in ("tc128", "skinny32", "pair256", "simt"):
        with pytest.raises(GstvdError) as e:
            eng.op_linear_ln(a, w, res=res, kernel=kernel)
        assert e.value.status == UNSUPPORTED, kernel
    with pytest.raises(GstvdError) as e:                 # whole 64-element k-chunks
        eng.op_linear_ln(torch.randn(M, 96), torch.randn(N, 96), res=res, kernel="ln32")
    assert e.value.status == UNSUPPORTED
    assert eng.launch_count == before


def test_matrix_names_match_header():
    assert set(GEMM_KERNELS) == {"simt", "tc32", "tc64", "tc128", "tc256", "skinny32", "skinny64", "pair128", "pair256", "ln32", "ln64"}
    assert GEMM_STORES == {"generic": 0, "tma": 1, "direct": 2}


# ---- engine integration: the cross K/V the prefill leaves for the decode kernels ------------------------------------------------
@pytest.fixture(scope="module")
def weighted(full_cfgs, full_sd):
    from gst_visdial_b200.engine import Engine
    enc_cfg, dec_cfg = full_cfgs
    engines = {}
    for dtype, mb in (("bf16", 64), ("fp32", 8)):
        e = Engine(enc_cfg, dec_cfg, device=0, dtype=dtype, max_batch=mb, max_beams=5)
        e.load_state_dict(full_sd)
        engines[dtype] = e
    yield engines
    for e in engines.values():
        e.close()


@pytest.mark.parametrize("dtype,B", [("bf16", 1), ("bf16", 8), ("bf16", 64), ("fp32", 3)])
def test_prefill_cross_cache(weighted, full_cfgs, full_sd, dtype, B):
    """prefill_cross on random fused states, read back: layer l, image b, row kv * heads + h holds (hidden @ W_kv^T + b) of that layer's
    cross-attention key (kv = 0) / value (kv = 1) weights, head h, in the [layer][image][kv * heads + h][Le][D] layout."""
    eng = weighted[dtype]
    dec = full_cfgs[1]
    H, heads, layers = dec.hidden_size, dec.num_attention_heads, dec.num_hidden_layers
    D, Le = H // heads, 293
    g = torch.Generator().manual_seed(B)
    hidden = torch.randn(B, Le, H, generator=g)
    eng.prefill_cross(B, Le, hidden, torch.ones(B, Le))
    cache = eng.debug_cross_cache(B, Le)
    x = (bf16(hidden) if dtype == "bf16" else hidden).cuda().double().reshape(B * Le, H)
    p = "decoder.decoder.bert.encoder.layer.{}.crossattention.self.{}.{}"
    for layer in range(layers):
        for kv, name in enumerate(("key", "value")):
            wt = full_sd[p.format(layer, name, "weight")].float()
            bt = full_sd[p.format(layer, name, "bias")].float().cuda().double()
            w64 = (bf16(wt) if dtype == "bf16" else wt).cuda().double()
            r = x @ w64.t() + bt
            mag = x.abs().sum(1, keepdim=True) * w64.abs().amax(1)[None, :]
            bound = H * U * mag + U * r.abs()
            if dtype == "bf16":
                bound = bound + ulp_bf16(r.abs() + bound)
            r = r.reshape(B, Le, heads, D).permute(0, 2, 1, 3)
            bound = bound.reshape(B, Le, heads, D).permute(0, 2, 1, 3)
            got = cache[layer, :, kv * heads:(kv + 1) * heads]
            what = f"prefill {dtype} B={B} layer {layer} {name}"
            assert bool(((got.double() - r).abs() <= bound).all()), what
    print(f"[gemm] prefill {dtype} B={B}: every layer within bound")
