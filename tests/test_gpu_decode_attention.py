"""GPU: the decode step's attention kernels one at a time against an fp64 reference of the same operation.

Every kernel runs through the single-kernel entries of the C ABI (gstvd_op_dec_self_attn, gstvd_op_dec_cross_attn,
gstvd_op_anc_update) on caller-supplied data, with the kernel forced instead of chosen by the environment.  The reference is fp64
softmax attention on the same (bf16-rounded) q / k / v, masked like the reference model, (1 - m) * -1e9; a query sees only its own
image's keys.  V is drawn from U(-1, 1), so |output| <= 1 and max-abs errors compare across cases.

Error model of the bf16 kernels (fp32 accumulation everywhere): the output is rounded to bf16 (relative 2^-9, at most ~2e-3 here);
the TMA and mma cross-attention kernels also round the un-normalised probabilities to bf16 before the P.V product (another 2^-9
relative per key) and the TMA kernels exponentiate with ex2.approx (~2^-22 relative).  The bounds below sit 2-3x above the largest
errors measured on a B200; the measured values are noted beside them.  fp32 kernels measured at most 5e-6 (logits of +-30), 1e-6
elsewhere.
"""
import math

import pytest
import torch

from helpers import max_abs, rel_rms

pytestmark = pytest.mark.gpu

TOL_F32 = 2e-5                           # max-abs of the fp32 kernels, as in test_gpu_ops.test_attention
# bf16 (rel-rms, max-abs) bounds; largest errors over every case of this file measured on a B200 (1000 W power limit) beside them.
# Kernels with fp32 probabilities err by the output rounding alone (max-abs 2^-9 = 1.95e-3 for |output| < 1); the TMA and mma kernels
# add the bf16 rounding of the probabilities.
TOL_BF16 = {
    "warp_tma": (4e-3, 8e-3),      # measured 1.54e-3, 3.04e-3
    "cta_tma": (4e-3, 8e-3),       # measured 1.54e-3, 3.04e-3
    "mma": (4e-3, 1e-2),           # measured 1.73e-3, 4.17e-3
    "simt": (3.5e-3, 5e-3),        # measured 1.32e-3, 1.95e-3
    "generic": (3.5e-3, 5e-3),     # measured 1.32e-3, 1.95e-3
    "v2": (4e-3, 5e-3),            # measured 1.70e-3, 1.95e-3
    "first": (4e-3, 5e-3),         # measured 1.70e-3, 1.95e-3
}


@pytest.fixture(scope="module")
def eng(full_cfgs):
    from gst_visdial_b200.engine import Engine
    enc_cfg, dec_cfg = full_cfgs
    e = Engine(enc_cfg, dec_cfg, device=0, dtype="bf16", max_batch=8, max_beams=5)
    yield e
    e.close()


def _round(t, dtype):
    return t.bfloat16().float() if dtype == "bf16" else t


def check_close(y, ref, kernel, dtype, what):
    y = y.cpu()
    assert torch.isfinite(y).all(), f"{what}: non-finite output"
    if dtype == "fp32":
        err = max_abs(y, ref)
        assert err < TOL_F32, f"{what}: max abs {err:.3e} (bound {TOL_F32})"
    else:
        rr, ma = rel_rms(y, ref), max_abs(y, ref)
        tol = TOL_BF16[kernel]
        assert rr < tol[0] and ma < tol[1], f"{what}: rel-rms {rr:.3e}, max-abs {ma:.3e} (bounds {tol})"


def same_bits(a, b):
    """Equal element for element, NaN matching NaN (stale cache rows hold NaN)."""
    return a.shape == b.shape and bool(((a == b) | (a.isnan() & b.isnan())).all())


# ---- cross-attention ---------------------------------------------------------------------------------------------------------
# (kernel, dtype, most keys it runs); the TMA kernels fetch at most five 64-key boxes and stop at 304 keys, the mma kernel at 320
CROSS_KERNELS = [("warp_tma", "bf16", 304), ("cta_tma", "bf16", 304), ("mma", "bf16", 320), ("simt", "bf16", 512), ("generic", "bf16", 512),
                 ("simt", "fp32", 512), ("generic", "fp32", 512)]
CROSS_LENS = [1, 15, 16, 17, 63, 64, 65, 128, 200, 293, 304, 320]   # 293: the real model (37 regions + 256 history tokens)
CROSS_K = [1, 2, 3, 5, 8]                                               # rows per image: every launch_cross_kb template
# last valid key + 1 of the history-shaped masks: either side of 16-key groups and 64-key boxes, cross_len % 16 == 1 included
HIST_LENS = (1, 2, 15, 16, 17, 31, 33, 37, 48, 63, 64, 65, 127, 128, 129, 192, 193, 255, 257, 289, 293, 300, 303, 305, 319)


def cross_masks(Le, seed):
    """One image per mask shape: all ones; history-shaped (valid prefix, padded tail) for every HIST_LENS entry below Le and Le - 1;
    holes among the first 37 keys (masked image regions) with and without a padded tail; only key 0 valid; every key masked."""
    g = torch.Generator().manual_seed(seed)
    ar = torch.arange(Le)
    rows = [torch.ones(Le)]
    rows += [(ar < n).float() for n in sorted({n for n in HIST_LENS if n < Le} | ({Le - 1} - {0}))]
    holes = (torch.rand(Le, generator=g) > 0.4).float()
    holes[37:] = 1.0
    holes[0] = 1.0
    rows.append(holes)
    if Le > 40:
        rows.append(holes * (ar < (Le + 37) // 2).float())
    rows.append((ar == 0).float())
    rows.append(torch.zeros(Le))
    return torch.stack(rows)


def cross_inputs(B, K, heads, Le, D, seed, q_scale=1.0):
    """q [B*K, heads*D] and cross K/V [B, 2*heads, Le, D] (k heads, then v heads); scores q.k / sqrt(D) have unit spread x q_scale."""
    g = torch.Generator().manual_seed(seed)
    q = torch.randn(B * K, heads * D, generator=g) * q_scale
    k = torch.randn(B, heads, Le, D, generator=g)
    v = torch.rand(B, heads, Le, D, generator=g) * 2 - 1
    return q, torch.cat([k, v], 1)


def ref_cross(q, kv, mask, K):
    """fp64 softmax(q k^T / sqrt(D) + (1 - m) * -1e9) v of every row over its own image's keys.
    A row whose keys are ALL masked follows the reference's fp32 arithmetic: there -1e9 swamps scores of a few units (the spacing of
    fp32 numbers near 1e9 is 64), every key gets the same weight and the result is the uniform mean of V.  fp64 would keep the raw
    scores' differences and give their softmax instead, which is not what the model computes."""
    B, two_heads, Le, D = kv.shape
    heads = two_heads // 2
    qh = q.double().view(B, K, heads, D).transpose(1, 2)                 # [B, heads, K, D]
    k, v = kv[:, :heads].double(), kv[:, heads:].double()                 # [B, heads, Le, D]
    s = qh @ k.transpose(-1, -2) / math.sqrt(D)
    if mask is not None:
        s = s + ((1.0 - mask.double()) * -1e9)[:, None, None, :]
    o = torch.softmax(s, -1) @ v
    if mask is not None:
        dead = (mask == 0).all(-1)
        o[dead] = v[dead].mean(-2, keepdim=True)
    return o.transpose(1, 2).reshape(B * K, heads * D)


def expected_cross_len(mask):
    """Last non-zero key + 1; Le for a row without one (the reference then spreads weight over every key)."""
    Le = mask.shape[1]
    last = torch.where(mask != 0, torch.arange(Le), torch.full_like(mask, -1, dtype=torch.long)).max(-1).values
    return torch.where(last < 0, torch.full_like(last, Le), last + 1)


def cross_case(eng, kernel, dtype, K, mask, q, kv, use_cross_len=True):
    """(kernel output, fp64 reference, cross_len or None) with q / kv rounded to the compute dtype first."""
    q, kv = _round(q, dtype), _round(kv, dtype)
    y, cl = eng.op_dec_cross_attn(q, kv, K, mask, use_cross_len=use_cross_len, kernel=kernel, dtype=dtype)
    return y.cpu(), ref_cross(q, kv, mask, K), (cl.cpu() if cl is not None else None)


CROSS_CASES = [(kernel, dtype, Le, K) for kernel, dtype, max_le in CROSS_KERNELS for Le in CROSS_LENS if Le <= max_le for K in CROSS_K]


@pytest.mark.parametrize("kernel,dtype,Le,K", CROSS_CASES)
def test_cross_attention(eng, kernel, dtype, Le, K):
    """Every mask shape of cross_masks at once (one image each, so the TMA kernels see a different cross_len per image)."""
    mask = cross_masks(Le, seed=Le)
    q, kv = cross_inputs(mask.shape[0], K, 12, Le, 64, seed=Le * 16 + K)
    y, ref, cl = cross_case(eng, kernel, dtype, K, mask, q, kv)
    check_close(y, ref, kernel, dtype, f"{kernel}/{dtype} Le={Le} K={K}")
    assert torch.equal(cl.long(), expected_cross_len(mask))


@pytest.mark.parametrize("kernel,dtype", [(k, d) for k, d, _ in CROSS_KERNELS])
@pytest.mark.parametrize("K", [1, 5])
def test_cross_attention_large_scores(eng, kernel, dtype, K):
    """Logits spanning about +-30: the maximum subtraction and the ex2.approx exponent of the TMA kernels at the sharp end.
    (No fully masked row here: a score of 30 is no longer swamped by -1e9 in fp32.)"""
    Le = 293
    mask = cross_masks(Le, seed=7)[:-1]
    q, kv = cross_inputs(mask.shape[0], K, 12, Le, 64, seed=99 + K, q_scale=10.0)
    y, ref, _ = cross_case(eng, kernel, dtype, K, mask, q, kv)
    s = _round(q, dtype).view(mask.shape[0], K, 12, 64)[:, :, 0] @ _round(kv, dtype)[:, 0].transpose(-1, -2) / 8.0
    assert s.abs().max() > 25.0, "the scores do not reach the intended range"
    check_close(y, ref, kernel, dtype, f"{kernel}/{dtype} large scores K={K}")


@pytest.mark.parametrize("kernel", [k for k, d, _ in CROSS_KERNELS if d == "bf16"])
def test_cross_attention_more_items_than_warp_slots(eng, kernel):
    """80 images x 12 heads = 960 (image, head) items, more than the 2 CTAs x 3 warps per SM of the warp-per-item kernel (and the
    2 CTAs per SM of the CTA-per-item kernel): slots loop over several items, so the box FIFO and the mbarrier phases carry over
    from one item to the next.  The images have different cross_len, so consecutive items fetch different numbers of boxes."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    B, heads, K, Le = 80, 12, 1, 293
    assert B * heads > 2 * sms * 3
    g = torch.Generator().manual_seed(80)
    lens = torch.randint(1, Le + 1, (B,), generator=g)
    lens[:10] = torch.tensor([1, 16, 17, 64, 65, 128, 129, 293, 200, 257])
    mask = (torch.arange(Le)[None, :] < lens[:, None]).float()
    mask[10:20, 1:37] *= (torch.rand(10, 36, generator=g) > 0.5).float()     # holes among the image regions
    mask[20] = 0.0                                                             # fully masked
    q, kv = cross_inputs(B, K, heads, Le, 64, seed=81)
    y, ref, cl = cross_case(eng, kernel, "bf16", K, mask, q, kv)
    check_close(y, ref, kernel, "bf16", f"{kernel} B={B} heads={heads}")
    assert torch.equal(cl.long(), expected_cross_len(mask))


@pytest.mark.parametrize("kernel", ["warp_tma", "cta_tma"])
@pytest.mark.parametrize("Le", [17, 65, 293, 304])
def test_cross_attention_tma_without_cross_len(eng, kernel, Le):
    """No key counts: the TMA kernels fetch all Le keys and the mask alone removes the padded tail."""
    mask = cross_masks(Le, seed=Le + 1)
    q, kv = cross_inputs(mask.shape[0], 3, 12, Le, 64, seed=Le + 2)
    y, ref, cl = cross_case(eng, kernel, "bf16", 3, mask, q, kv, use_cross_len=False)
    assert cl is None
    check_close(y, ref, kernel, "bf16", f"{kernel} Le={Le} without cross_len")


@pytest.mark.parametrize("kernel", ["default", "generic"])
@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("Le", [1, 17, 293, 512])
def test_cross_attention_head_dim_128(eng, kernel, dtype, Le):
    """128-dim heads: only the generic kernel runs them (the decode step's own choice too)."""
    mask = cross_masks(Le, seed=Le + 3)
    q, kv = cross_inputs(mask.shape[0], 2, 6, Le, 128, seed=Le + 4)
    y, ref, _ = cross_case(eng, kernel, dtype, 2, mask, q, kv)
    check_close(y, ref, "generic", dtype, f"{kernel}/{dtype} D=128 Le={Le}")


@pytest.mark.parametrize("Le", [1, 31, 32, 33, 293, 512])
def test_cross_len(eng, Le):
    """cross_len_kernel: last non-zero mask entry + 1, Le for an all-zero row; non-binary entries count as non-zero."""
    B = 37
    g = torch.Generator().manual_seed(Le)
    mask = (torch.rand(B, Le, generator=g) > 0.6).float()
    tails = torch.randint(0, Le + 1, (B,), generator=g)
    mask *= (torch.arange(Le)[None, :] < tails[:, None]).float()
    mask[0] = 0.0
    mask[1] = 1.0
    mask[2] = 0.0
    mask[2, 0] = 1.0
    mask[3] = 0.0
    mask[3, Le - 1] = 0.5
    q, kv = cross_inputs(B, 1, 2, Le, 64, seed=Le + 5)
    y, ref, cl = cross_case(eng, "simt", "fp32", 1, mask, q, kv)
    assert torch.equal(cl.long(), expected_cross_len(mask)), (cl, expected_cross_len(mask))
    check_close(y, ref, "simt", "fp32", f"cross_len Le={Le}")


def test_forced_kernels_refuse_unsupported_shapes(eng):
    """A forced kernel outside its range is refused before anything runs (GSTVD_ERR_UNSUPPORTED), never replaced by another."""
    from gst_visdial_b200._lib import GstvdError
    for kernel, dtype, Le, D in (("warp_tma", "bf16", 305, 64), ("cta_tma", "fp32", 64, 64), ("mma", "bf16", 321, 64),
                                 ("mma", "bf16", 64, 128), ("simt", "fp32", 64, 128)):
        q, kv = cross_inputs(1, 1, 2, Le, D, seed=1)
        with pytest.raises(GstvdError) as e:
            eng.op_dec_cross_attn(q, kv, 1, None, use_cross_len=False, kernel=kernel, dtype=dtype)
        assert e.value.status == -3, (kernel, dtype, Le, D)
    H = 768
    qkv, cache = torch.randn(5, 3 * H), torch.zeros(2, 1, 18, 5, H)
    for kernel, dtype, anc in (("v2", "fp32", None), ("first", "bf16", torch.zeros(5, 32, dtype=torch.uint8))):
        with pytest.raises(GstvdError) as e:
            eng.op_dec_self_attn(qkv, cache, 12, step=0, anc=anc, kernel=kernel, dtype=dtype)
        assert e.value.status == -3, (kernel, dtype)


# ---- self-attention ----------------------------------------------------------------------------------------------------------
# (kernel, dtype, head_dim, ancestry table); the first kernel is the fp32 path and the GSTVD_SELF_V2=0 path of bf16
SELF_KERNELS = [("v2", "bf16", 64, False), ("v2", "bf16", 64, True), ("first", "bf16", 64, False), ("first", "bf16", 128, False),
                ("first", "fp32", 64, False), ("first", "fp32", 128, False)]
# T <= 20 / <= 32 / <= 64: the NIT = 5 / 8 / 16 lean kernels, NS = 1 / 2 of the first kernel, ancestry rows of 32 / 64 entries
SELF_T = [18, 20, 21, 32, 33, 64]
SELF_P0 = [0, 1, 7, 25]


def self_cases():
    out = []
    for T in SELF_T:
        for P0 in SELF_P0:
            if P0 >= T:
                continue
            for step in sorted({0, (T - P0 - 1) // 2, T - P0 - 1}):
                out.append((T, P0, step))
    return out


def self_inputs(B, K, heads, D, T, P0, step, seed, dtype, with_anc, with_prefix):
    """qkv [B*K, 3H]; cache [2, B, T, K, H] with NaN at and past the new position in every slot (cudaMalloc memory is not zeroed:
    the kernels must never let those rows into the result); prefix_qkv [B*P0, 3H] or None; anc uint8 [B*K, 32 or 64] with repeated
    parents below the new position and stale entries >= K from it on, or None."""
    g = torch.Generator().manual_seed(seed)
    H, pos = heads * D, P0 + step
    qkv = torch.cat([torch.randn(B * K, H, generator=g), torch.randn(B * K, H, generator=g), torch.rand(B * K, H, generator=g) * 2 - 1], 1)
    cache = torch.stack([torch.randn(B, T, K, H, generator=g), torch.rand(B, T, K, H, generator=g) * 2 - 1])
    cache[:, :, pos:] = float("nan")
    prefix = None
    if with_prefix:
        prefix = torch.cat([torch.randn(B * P0, H, generator=g), torch.randn(B * P0, H, generator=g),
                            torch.rand(B * P0, H, generator=g) * 2 - 1], 1)
    anc = None
    if with_anc:
        W = 32 if T <= 32 else 64
        anc = torch.randint(0, K, (B * K, W), generator=g)
        anc[:, pos:] = torch.randint(K, 256, (B * K, W - pos), generator=g)
        anc = anc.to(torch.uint8)
    r = lambda t: None if t is None else _round(t, dtype)
    return r(qkv), r(cache), r(prefix), anc


def ref_self_cache(qkv, cache, prefix, B, K, P0, step):
    """The cache after the call: the input, the prefix rows in positions 0..P0-1 of every slot, the new k / v at P0 + step of each
    row's own slot."""
    H = cache.shape[-1]
    exp = cache.clone()
    if prefix is not None:
        pk = prefix.view(B, P0, 3, H)
        exp[0, :, :P0] = pk[:, :, 1, None, :]
        exp[1, :, :P0] = pk[:, :, 2, None, :]
    q3 = qkv.view(B, K, 3, H)
    exp[0, :, P0 + step] = q3[:, :, 1]
    exp[1, :, P0 + step] = q3[:, :, 2]
    return exp


def ref_self_attn(qkv, cache_after, anc, B, K, heads, P0, step):
    """fp64 attention of each row's new query over its history: position t < P0 + step from slot anc[b*K + k, t] (own slot without a
    table), position P0 + step its own new k / v."""
    H = cache_after.shape[-1]
    D, pos = H // heads, P0 + step
    if anc is None:
        slot = torch.arange(K)[None, :, None].expand(B, K, pos)
    else:
        slot = anc.view(B, K, -1)[:, :, :pos].long()
    bi, ti = torch.arange(B)[:, None, None], torch.arange(pos)[None, None, :]
    q3 = qkv.view(B, K, 3, H)
    keys = torch.cat([cache_after[0][bi, ti, slot], q3[:, :, 1, None]], 2).double().view(B, K, pos + 1, heads, D)
    vals = torch.cat([cache_after[1][bi, ti, slot], q3[:, :, 2, None]], 2).double().view(B, K, pos + 1, heads, D)
    q = q3[:, :, 0].double().view(B, K, heads, D)
    p = torch.softmax(torch.einsum("bkhd,bkthd->bkht", q, keys) / math.sqrt(D), -1)
    return torch.einsum("bkht,bkthd->bkhd", p, vals).reshape(B * K, H)


def self_case(eng, kernel, dtype, D, with_anc, T, P0, step, step_known):
    """(output, reference, cache after the call, expected cache).  P0 = 1 and 25 store a prefix first (prefix_kv_store); P0 = 7 keeps
    per-slot prefix rows from the caller's cache."""
    B, K, heads = 3, (8 if with_anc else 5), 768 // D
    qkv, cache, prefix, anc = self_inputs(B, K, heads, D, T, P0, step, T * 1000 + P0 * 100 + step * 3 + D, dtype, with_anc, P0 in (1, 25))
    y, c = eng.op_dec_self_attn(qkv, cache, heads, P0=P0, step=step, step_known=step_known, prefix_qkv=prefix, anc=anc, kernel=kernel,
                                dtype=dtype)
    exp = ref_self_cache(qkv, cache, prefix, B, K, P0, step)
    return y.cpu(), ref_self_attn(qkv, exp, anc, B, K, heads, P0, step), c.cpu(), exp


@pytest.mark.parametrize("kernel,dtype,D,with_anc", SELF_KERNELS)
@pytest.mark.parametrize("T,P0,step", self_cases())
def test_self_attention(eng, kernel, dtype, D, with_anc, T, P0, step):
    for step_known in (True, False):
        y, ref, c, exp = self_case(eng, kernel, dtype, D, with_anc, T, P0, step, step_known)
        what = f"{kernel}/{dtype} D={D} anc={with_anc} T={T} P0={P0} step={step} step_known={step_known}"
        check_close(y, ref, kernel, dtype, what)
        assert same_bits(c, exp), f"{what}: the cache differs from the input + prefix rows + appended k/v"


@pytest.mark.parametrize("T,P0", [(18, 0), (40, 7)])
def test_self_attention_beam_chain(eng, T, P0):
    """A whole beam search's self-attention: every step, random parents (repeats included).  Three paths must agree:
    (a) the lean kernel reading through the ancestry table, updated by anc_update_kernel, the cache never moved;
    (b) the first kernel with the reorder_cache semantics, index_select of the cache over the beams after every step;
    (c) the fp64 reference over the gathered history.
    The table itself is checked against the host rule of test_beam_oracle.test_ancestry_table_equals_cache_gather."""
    B, K, heads, D = 3, 5, 12, 64
    H, W = heads * D, (32 if T <= 32 else 64)
    g = torch.Generator().manual_seed(T + P0)
    dev = eng.device
    cache_a = torch.full((2, B, T, K, H), float("nan"), device=dev)
    cache_b = cache_a.clone()
    ref_cache = torch.full((2, B, T, K, H), float("nan"))               # held on the host, gathered like (b)
    anc = torch.randint(0, 256, (B * K, W), generator=g).to(torch.uint8)  # never written yet: stale everywhere
    anc_ref = anc.clone()
    prefix = None
    if P0 > 0:
        prefix = _round(torch.cat([torch.randn(B * P0, H, generator=g), torch.randn(B * P0, H, generator=g),
                                   torch.rand(B * P0, H, generator=g) * 2 - 1], 1), "bf16")
    bi, kk = torch.arange(B)[:, None], torch.arange(K)[None, :]
    for step in range(T - P0):
        pos = P0 + step
        qkv = _round(torch.cat([torch.randn(B * K, H, generator=g), torch.randn(B * K, H, generator=g),
                                torch.rand(B * K, H, generator=g) * 2 - 1], 1), "bf16")
        pre = prefix if step == 0 else None
        y_a, cache_a = eng.op_dec_self_attn(qkv, cache_a, heads, P0=P0, step=step, prefix_qkv=pre, anc=anc, kernel="v2", dtype="bf16")
        y_b, cache_b = eng.op_dec_self_attn(qkv, cache_b, heads, P0=P0, step=step, prefix_qkv=pre, kernel="first", dtype="bf16")
        ref_cache = ref_self_cache(qkv, ref_cache, pre, B, K, P0, step)
        ref = ref_self_attn(qkv, ref_cache, None, B, K, heads, P0, step)
        check_close(y_a.cpu(), ref, "v2", "bf16", f"(a) ancestry path, T={T} P0={P0} step={step}")
        check_close(y_b.cpu(), ref, "first", "bf16", f"(b) gather path, T={T} P0={P0} step={step}")
        assert same_bits(cache_b.cpu(), ref_cache), f"step {step}: gathered cache"
        # (a) never moves rows: the history of beam k is in slot anc[k][t] (prefix rows are in every slot, whatever the stale entry says)
        ca = cache_a.cpu()
        slot = anc_ref.view(B, K, W)[:, :, :pos + 1].long().clamp(max=K - 1)
        assert (anc_ref.view(B, K, W)[:, :, P0:pos].long() < K).all(), f"step {step}: unwritten ancestry entry inside the history"
        slot[:, :, pos] = kk
        ti = torch.arange(pos + 1)[None, None, :]
        hist_a = ca[:, bi[:, :, None], ti, slot]                         # [2, B, K, pos + 1, H]
        assert same_bits(hist_a, ref_cache[:, :, :pos + 1].transpose(2, 3)), f"step {step}: ancestry reads differ from the gather"
        # beam selection
        parent = torch.randint(0, K, (B, K), generator=g)
        anc = eng.op_anc_update(anc, parent, T, P0, step).cpu()
        new = anc_ref.view(B, K, W).clone()
        new[:, :, :pos] = anc_ref.view(B, K, W)[bi, parent, :pos]
        new[:, :, pos] = parent.to(torch.uint8)
        anc_ref = new.view(B * K, W)
        assert torch.equal(anc, anc_ref), f"step {step}: ancestry table"
        cache_b = cache_b[:, bi.to(dev), :, parent.to(dev)].permute(2, 0, 3, 1, 4).contiguous()
        ref_cache = ref_cache[:, bi, :, parent].permute(2, 0, 3, 1, 4).contiguous()
