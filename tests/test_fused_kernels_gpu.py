"""The fused 16-bit kernels called on their own (lib.attention_fwd/bwd, lib.ffn_fwd/bwd) against float64 references
computed from the same 16-bit operands the kernels read, in bf16 and fp16.

Errors are measured per row (max-abs error of each (b, h, query row) / key row / FFN row, divided by that row's reference
scale) and as a global relative L2, so that a bug confined to one tile, one key block or one hidden slice cannot be
averaged away.  Bounds follow from the roundings the kernels do, with u the unit roundoff of the 16-bit type
(2^-8 bf16, 2^-11 fp16).  Beside each bound: the worst per-row error as a fraction of it, bf16 / fp16, measured on a
B200 (1000 W power limit, 1965 MHz max SM clock) over this file's cases:
  ctx     : P rounded to 16 bits before PV, ctx rounded           -> 2u of sum_k |P_k| |V_k|              0.55 / 0.56
  lse     : fp32 logits, ex2.approx, fp32 row sum                 -> 1e-4 + 2^-20 |lse|                   0.007 / 0.008
  dV      : P rounded before dV = P^T dO, dV rounded              -> 2u of |P|^T |dO|                     0.75 / 0.73
  dQ, dK  : dS rounded before the two products, output rounded,
            D = rowsum(dO * O) taken from the 16-bit O            -> 2u of (|dS| + P D_abs) |K| (|Q|)     dQ 0.28 / 0.33, dK 0.57 / 0.58
  F1, dF1 : one rounding of an fp32 value to 16 bits              -> u + 2^-14 of the row's magnitude     F1 0.45 / 0.40, dF1 0.45 / 0.42
  x_out, dH: fp32 accumulation only (the reference takes the kernel's own 16-bit F1 / dF1 as the GEMM input)
                                                                  -> 2^-14 of the row's magnitude         x_out 0.008 / 0.013, dH 0.008 / 0.011
fp16 adds an absolute term for subnormal flushing of small P / dS / activations (2^-25 per element of a contraction).
The global L2 errors measured at most 0.17 of the same bounds.  The whole file runs in about 6 s on a B200.
"""
import math

import numpy
import pytest
import torch

from neurst_b200 import lib as L

pytestmark = pytest.mark.gpu

DTYPES = {"bf16": (torch.bfloat16, 2.0 ** -8), "fp16": (torch.float16, 2.0 ** -11)}
MASK_MIN = -1.0e9
FP32_SLACK = 2.0 ** -14        # fp32 accumulation in the tensor core and the slice reduce-add, relative to the row scale
SENTINEL = 1000.0
WORST = {}                     # (check, dtype) -> worst per-row error / bound, printed at the end of the module


def _note(name, dt, ratio):
    key = (name, dt)
    WORST[key] = max(WORST.get(key, 0.0), ratio)


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for (name, dt), r in sorted(WORST.items()):
        print("worst %-12s %s: %.3f of the bound" % (name, dt, r))


def _tiny(dt):
    return 2.0 ** -25 if dt == "fp16" else 0.0


def _row_check(name, dt, got, ref, scale, bound, absterm=0.0):
    """max_row |got - ref| <= bound * scale_row + absterm for every row (rows along dim 0 after flattening the rest), and
    globally ||got - ref||_2 <= bound * ||scale||_2 + absterm.  The global L2 is taken relative to the scale, the magnitude
    the rounding errors are proportional to, not to ||ref||: dQ cancels (sum_k dS = 0 in every row; it is exactly 0 for a
    single key), so its own norm can sit below the rounding noise."""
    diff = got.double() - ref
    err = diff.abs().reshape(ref.shape[0], -1).amax(1)
    lim = bound * scale.reshape(ref.shape[0], -1).amax(1) + absterm + 1e-30
    ratio = float((err / lim).max())
    _note(name, dt, ratio)
    assert ratio <= 1.0, "%s: per-row error %.3g x the bound (row %d)" % (name, ratio, int((err / lim).argmax()))
    l2 = float(diff.norm() / (bound * scale.double().norm() + absterm + 1e-30))
    _note(name + " L2", dt, l2)
    assert l2 <= 1.0, "%s: global L2 error %.3g x the bound" % (name, l2)
    return ratio


def _worst_ratio(got, ref, scale, bound, absterm=0.0):
    err = (got.double() - ref).abs().reshape(ref.shape[0], -1).amax(1)
    lim = bound * scale.reshape(ref.shape[0], -1).amax(1) + absterm + 1e-30
    return float((err / lim).max())


def _keep_bits(n, p, seed, stream):
    """(packed keep bitmap uint8 [n/8] on the device, keep mask bool [n] on the device) of b200st_dropout_mask."""
    m = torch.empty(n, dtype=torch.uint8, device="cuda")
    L.check(L.load().b200st_dropout_mask(seed, stream, n, p, m.data_ptr(), L._stream()))
    packed = numpy.packbits(m.cpu().numpy(), bitorder="little")
    return torch.from_numpy(packed).cuda(), m.bool()


def _sentinel_ok(buf, before, view_mask):
    """every element outside view_mask still holds its initial bits"""
    same = buf.view(torch.int16 if buf.element_size() == 2 else torch.int32) == before
    return bool(same[~view_mask].all())


# ---------------------------------------------------------------------------------------------------------------------
# attention
# ---------------------------------------------------------------------------------------------------------------------
def _attn_reference(q, k, v, B, H, Tq, Tk, bias, causal, keep, scale_p, causal_shift=0):
    """float64 P (with the fp32 rule for fully masked rows), dropped P, ctx, lse.  q: [B*Tq, H*64] 16-bit."""
    Q = q.double().reshape(B, Tq, H, 64).permute(0, 2, 1, 3)
    K = k.double().reshape(B, Tk, H, 64).permute(0, 2, 1, 3)
    V = v.double().reshape(B, Tk, H, 64).permute(0, 2, 1, 3)
    logits = Q @ K.transpose(-1, -2) * 0.125
    if bias is not None:
        logits = logits + bias.double()[:, None, None, :]
    if causal:
        kk = torch.arange(Tk, device=q.device)[None, :]
        qq = torch.arange(Tq, device=q.device)[:, None]
        logits = logits + torch.where(kk > qq + (Tk - Tq) + causal_shift, MASK_MIN, 0.0).double()
    lse = torch.logsumexp(logits, -1)
    P = torch.softmax(logits, -1)
    if bias is not None:
        # every key biased by -1e9: in fp32, -1e9 + s rounds to -1e9 for every key, so the row is uniform over all Tk keys
        full = (bias <= MASK_MIN).all(1)
        P[full] = 1.0 / Tk
    Pd = P * keep.double() * scale_p if keep is not None else P
    ctx = Pd @ V
    return Q, K, V, P, Pd, ctx, lse


ATTN_CASES = [
    # (B, H, Tq, Tk, causal, bias lengths (None: no bias; 0 = fully padded), pass kv_len, dropout p, ctx column padding)
    (1, 1, 1, 1, False, None, False, 0.0, 0),
    (2, 4, 64, 64, False, None, False, 0.1, 64),
    (2, 4, 127, 127, False, [127, 1], True, 0.0, 0),
    (3, 8, 128, 128, False, [128, 127, 1], False, 0.1, 0),
    (2, 4, 129, 129, False, [128, 129], True, 0.1, 8),
    (3, 4, 250, 250, False, [0, 129, 250], True, 0.1, 0),
    (2, 8, 375, 375, False, [128, 375], True, 0.0, 0),
    (3, 8, 750, 750, False, [129, 750, 1], True, 0.1, 0),
    (1, 4, 750, 750, False, None, False, 0.0, 0),
    (3, 4, 9, 250, False, [250, 127, 1], True, 0.1, 0),
    (2, 8, 88, 250, False, [0, 129], True, 0.0, 0),
    (2, 4, 128, 375, False, [375, 128], False, 0.1, 0),
    (3, 8, 152, 750, False, [750, 129, 127], True, 0.1, 64),
    (2, 4, 9, 9, True, None, False, 0.1, 0),
    (3, 8, 88, 88, True, None, False, 0.1, 0),
    (2, 4, 128, 128, True, None, False, 0.0, 0),
    (1, 1, 129, 129, True, None, False, 0.1, 0),
    (2, 8, 300, 300, True, None, False, 0.1, 0),
]


def _case_id(c):
    B, H, Tq, Tk, causal, lens, kvl, p, pad = c
    return "B%dH%d_%dx%d%s%s%s_p%g" % (B, H, Tq, Tk, "_causal" if causal else "", "" if lens is None else "_bias",
                                      "_kvlen" if kvl else "", p)


@pytest.mark.parametrize("dt", list(DTYPES))
@pytest.mark.parametrize("case", ATTN_CASES, ids=_case_id)
def test_fused_attention_matches_fp64(case, dt):
    B, H, Tq, Tk, causal, lens, pass_kvlen, p, ctx_pad = case
    tdt, u = DTYPES[dt]
    dev = "cuda"
    g = torch.Generator(device=dev).manual_seed(1000 * Tq + Tk + 7 * B + H)
    HD = H * 64
    self_attn = Tq == Tk
    pad_rows = 5
    # operands as column views of the packed projections the model passes: [B*T, 3*H*64] (self) or q + [B*Tk, 2*H*64]
    if self_attn:
        qkv = (torch.randn(B * Tq + pad_rows, 3 * HD, generator=g, device=dev)).to(tdt)
        q, k, v = qkv[:B * Tq, :HD], qkv[:B * Tk, HD:2 * HD], qkv[:B * Tk, 2 * HD:]
    else:
        qb = torch.randn(B * Tq + pad_rows, HD, generator=g, device=dev).to(tdt)
        kv = torch.randn(B * Tk + pad_rows, 2 * HD, generator=g, device=dev).to(tdt)
        q, k, v = qb[:B * Tq], kv[:B * Tk, :HD], kv[:B * Tk, HD:]
    bias = kv_len = None
    if lens is not None:
        bias = torch.zeros(B, Tk, device=dev)
        for b, n in enumerate(lens):
            bias[b, n:] = MASK_MIN
        if pass_kvlen:
            kv_len = torch.tensor([n if n > 0 else Tk for n in lens], dtype=torch.int32, device=dev)
    Tkp = (Tk + 7) // 8 * 8
    keep = bits = None
    if p > 0:
        bits, mask = _keep_bits(B * H * Tq * Tkp, p, 1234 + Tk, 77 + Tq)
        keep = mask.reshape(B, H, Tq, Tkp)[..., :Tk]
    scale_p = 1.0 / (1.0 - p) if p > 0 else 1.0

    ctx_buf = torch.full((B * Tq + pad_rows, HD + ctx_pad), SENTINEL, dtype=tdt, device=dev)
    ctx_before = ctx_buf.view(torch.int16).clone()
    ctx = ctx_buf[:B * Tq, :HD]
    lse = torch.full((B, H, Tq), SENTINEL, device=dev)
    L.attention_fwd(q, k, v, ctx, lse, B, H, bias=bias, kv_len=kv_len, causal=causal, drop_p=p, keep_bits=bits)
    torch.cuda.synchronize()

    Q, K, V, P, Pd, ctx_ref, lse_ref = _attn_reference(q, k, v, B, H, Tq, Tk, bias, causal, keep, scale_p)
    got_ctx = ctx.double().reshape(B, Tq, H, 64).permute(0, 2, 1, 3)
    ctx_scale = Pd @ V.abs()
    sub = _tiny(dt) * Tk * V.abs().amax() * scale_p
    # ctx: 2u (P and ctx roundings)
    _row_check("ctx", dt, got_ctx.reshape(-1, 64), ctx_ref.reshape(-1, 64), ctx_scale.reshape(-1, 64), 2 * u, float(sub))
    # lse: fp32 logits, ex2.approx and an fp32 row sum: 1e-4 absolute + 2^-20 relative (fully padded rows sit at -1e9)
    lse_err = (lse.double() - lse_ref).abs()
    lse_lim = 1e-4 + 2.0 ** -20 * lse_ref.abs()
    _note("lse", dt, float((lse_err / lse_lim).max()))
    assert bool((lse_err <= lse_lim).all()), float((lse_err / lse_lim).max())
    view = torch.zeros_like(ctx_buf, dtype=torch.bool)
    view[:B * Tq, :HD] = True
    assert _sentinel_ok(ctx_buf, ctx_before, view), "fused attention forward wrote outside the ctx view"

    # ---- the reference must reject a kernel with a plausible bug: each mutation moves ctx by > 5x the bound ----
    def mutated_ratio(**kw):
        args = dict(bias=bias, causal=causal, keep=keep)
        args.update(kw)
        m = _attn_reference(q, k, v, B, H, Tq, Tk, args["bias"], args["causal"], args["keep"], scale_p,
                            causal_shift=kw.get("causal_shift", 0))[5]
        return _worst_ratio(got_ctx.reshape(-1, 64), m.reshape(-1, 64), ctx_scale.reshape(-1, 64), 2 * u, float(sub))

    if causal and Tq > 1:
        assert mutated_ratio(causal_shift=1) > 5, "a causal mask shifted by one key passes the ctx bound"
    if kv_len is not None and min(lens) > 0:
        assert mutated_ratio(bias=torch.zeros_like(bias)) > 5, "an unpadded kv_len tail passes the ctx bound"
    if keep is not None:
        shifted = torch.roll(mask, 1).reshape(B, H, Tq, Tkp)[..., :Tk]
        assert mutated_ratio(keep=shifted) > 5, "a dropout bitmap shifted by one element passes the ctx bound"

    # ---- backward ----
    dO = torch.randn(B * Tq, HD, generator=g, device=dev).to(tdt)
    if self_attn:
        dbuf = torch.full((B * Tq + pad_rows, 3 * HD), SENTINEL, dtype=tdt, device=dev)
        dq, dk, dv = dbuf[:B * Tq, :HD], dbuf[:B * Tk, HD:2 * HD], dbuf[:B * Tk, 2 * HD:]
        bufs = [(dbuf, [(slice(0, B * Tq), slice(0, 3 * HD))])]
    else:
        dqb = torch.full((B * Tq + pad_rows, HD + 64), SENTINEL, dtype=tdt, device=dev)
        dkvb = torch.full((B * Tk + pad_rows, 2 * HD), SENTINEL, dtype=tdt, device=dev)
        dq, dk, dv = dqb[:B * Tq, :HD], dkvb[:B * Tk, :HD], dkvb[:B * Tk, HD:]
        bufs = [(dqb, [(slice(0, B * Tq), slice(0, HD))]), (dkvb, [(slice(0, B * Tk), slice(0, 2 * HD))])]
    befores = [b.view(torch.int16).clone() for b, _ in bufs]
    scratch = torch.empty(B * Tq * HD + B * H * Tq, device=dev)
    L.attention_bwd(q, k, v, ctx, dO, lse, dq, dk, dv, scratch, B, H, bias=bias, kv_len=kv_len, causal=causal, drop_p=p,
                    keep_bits=bits)
    torch.cuda.synchronize()

    dOr = dO.double().reshape(B, Tq, H, 64).permute(0, 2, 1, 3)
    O16 = got_ctx
    kd = keep.double() * scale_p if keep is not None else 1.0
    dV_ref = Pd.transpose(-1, -2) @ dOr
    dPd = (dOr @ V.transpose(-1, -2)) * kd
    Dvec = (dOr * ctx_ref).sum(-1, keepdim=True)
    dS = P * (dPd - Dvec)
    dQ_ref = dS @ K * 0.125
    dK_ref = dS.transpose(-1, -2) @ Q * 0.125
    D_abs = (dOr.abs() * O16.abs()).sum(-1, keepdim=True)
    dS_scale = dS.abs() + P * D_abs
    sub_s = _tiny(dt)
    # dV: 2u (P and dV roundings)
    _row_check("dV", dt, dv.double().reshape(B, Tk, H, 64).permute(0, 2, 1, 3).reshape(-1, 64), dV_ref.reshape(-1, 64),
               (Pd.transpose(-1, -2) @ dOr.abs()).reshape(-1, 64), 2 * u, float(sub_s * Tq * dOr.abs().amax() * scale_p))
    # dQ, dK: 2u (dS and output roundings, D from the 16-bit O folded into the scale)
    _row_check("dQ", dt, dq.double().reshape(B, Tq, H, 64).permute(0, 2, 1, 3).reshape(-1, 64), dQ_ref.reshape(-1, 64),
               (dS_scale @ K.abs() * 0.125).reshape(-1, 64), 2 * u, float(sub_s * Tk * K.abs().amax() * 0.125))
    _row_check("dK", dt, dk.double().reshape(B, Tk, H, 64).permute(0, 2, 1, 3).reshape(-1, 64), dK_ref.reshape(-1, 64),
               (dS_scale.transpose(-1, -2) @ Q.abs() * 0.125).reshape(-1, 64), 2 * u,
               float(sub_s * Tq * Q.abs().amax() * 0.125))
    for (b, views), before in zip(bufs, befores):
        view = torch.zeros_like(b, dtype=torch.bool)
        for rs, cs in views:
            view[rs, cs] = True
        assert _sentinel_ok(b, before, view), "fused attention backward wrote outside the dq / dk / dv views"


def test_fused_attention_refuses_bad_arguments():
    dev = "cuda"
    x = torch.zeros(128, 64, dtype=torch.bfloat16, device=dev)
    lse = torch.zeros(1, 1, 128, device=dev)
    with pytest.raises(L.B200STError, match="keep bitmap"):
        L.attention_fwd(x, x, x, x.clone(), lse, 1, 1, drop_p=0.1)
    with pytest.raises(L.B200STError, match="16-bit"):
        L.attention_fwd(x.float(), x.float(), x.float(), x.float(), lse, 1, 1)
    lib = L.load()
    with pytest.raises(L.B200STError, match="null"):
        L.check(lib.b200st_attention_fwd(L.BF16, None, 64, x.data_ptr(), 64, x.data_ptr(), 64, 1, 1, 128, 128, None, None, 0,
                                         0.0, None, x.data_ptr(), 64, lse.data_ptr(), L._stream()))


# ---------------------------------------------------------------------------------------------------------------------
# FFN
# ---------------------------------------------------------------------------------------------------------------------
FFN_SHAPES = [(128, 1), (128, 129), (128, 19000), (512, 128), (512, 1000), (512, 2816), (512, 8000), (2048, 100),
              (2048, 129), (2048, 1000), (2048, 2816), (2048, 8000), (2048, 19000)]
SPLITS_SEEN = set()


@pytest.mark.parametrize("dt", list(DTYPES))
@pytest.mark.parametrize("d", [128, 256])
@pytest.mark.parametrize("ffn,M", FFN_SHAPES, ids=["ffn%d_M%d" % s for s in FFN_SHAPES])
def test_fused_ffn_matches_fp64(ffn, M, d, dt):
    tdt, u = DTYPES[dt]
    dev = "cuda"
    g = torch.Generator(device=dev).manual_seed(M * 7 + ffn + d)
    p = 0.1 if (FFN_SHAPES.index((ffn, M)) + d // 128) % 2 else 0.0
    pad_rows = 3
    X = torch.randn(M, d, generator=g, device=dev).to(tdt)
    W1 = (torch.randn(d, ffn, generator=g, device=dev) / math.sqrt(d)).to(tdt)
    W2 = (torch.randn(ffn, d, generator=g, device=dev) / math.sqrt(ffn)).to(tdt)
    b1 = torch.randn(ffn, generator=g, device=dev) * 0.5
    b2 = torch.randn(d, generator=g, device=dev) * 0.5
    resid = torch.randn(M, d, generator=g, device=dev)
    fbits = pbits = None
    fscale = pscale = 1.0
    fkeep = pkeep = torch.ones(1, device=dev, dtype=torch.bool)
    if p > 0:
        fbits, fkeep = _keep_bits(M * ffn, p, 99 + M, 5)
        pbits, pkeep = _keep_bits(M * d, p, 98 + M, 6)
        fkeep, pkeep = fkeep.reshape(M, ffn), pkeep.reshape(M, d)
        fscale = pscale = 1.0 / (1.0 - p)

    F1b = torch.full((M + pad_rows, ffn), SENTINEL, dtype=tdt, device=dev)
    xb = torch.full((M + pad_rows, d), SENTINEL, device=dev)
    xb[:M] = resid
    splits = L.ffn_fwd(X, W1, b1, W2, b2, F1b, xb, drop_ffn_p=p, ffn_bits=fbits, drop_post_p=p, post_bits=pbits)
    SPLITS_SEEN.add((splits, ffn // 128))
    torch.cuda.synchronize()
    F1, x_out = F1b[:M], xb[:M]

    Xd, W1d, W2d = X.double(), W1.double(), W2.double()
    Hd = Xd @ W1d + b1.double()
    F1_ref = torch.relu(Hd) * fkeep.double() * fscale
    F1_scale = (Xd.abs() @ W1d.abs() + b1.double().abs()) * fscale
    # F1: one rounding of the fp32 activation (u) + fp32 accumulation slack
    _row_check("F1", dt, F1, F1_ref, F1_scale, u + FP32_SLACK, _tiny(dt))
    # x_out from the kernel's own 16-bit hidden activations: fp32 accumulation only
    F1k = F1.double()
    y = F1k @ W2d + b2.double()
    x_ref = resid.double() + y * pkeep.double() * pscale
    x_scale = (F1k.abs() @ W2d.abs() + b2.double().abs()) * pscale + resid.double().abs()
    _row_check("x_out", dt, x_out, x_ref, x_scale, FP32_SLACK)
    assert bool((xb[M:] == SENTINEL).all()) and bool((F1b[M:] == SENTINEL).all()), "rows >= M written"
    # the bound rejects b2 added on every slice / twice and a hidden slice left out
    assert _worst_ratio(x_out, x_ref + b2.double() * pkeep.double() * pscale, x_scale, FP32_SLACK) > 5
    chunks = ffn // 128
    drop_cols = slice((chunks // splits) * 128 * (splits - 1), ffn) if splits > 1 else slice(0, 128)
    if splits > 1 or chunks > 1:
        F1_miss = F1k.clone()
        F1_miss[:, drop_cols] = 0
        miss_ref = resid.double() + (F1_miss @ W2d + b2.double()) * pkeep.double() * pscale
        assert _worst_ratio(x_out, miss_ref, x_scale, FP32_SLACK) > 5

    # ---- data gradient ----
    dY = torch.randn(M, d, generator=g, device=dev).to(tdt)
    dF1b = torch.full((M + pad_rows, ffn), SENTINEL, dtype=tdt, device=dev)
    dHb = torch.full((M + pad_rows, d), SENTINEL, device=dev)
    dH0 = torch.randn(M, d, generator=g, device=dev)
    dHb[:M] = dH0
    bsplits = L.ffn_bwd(dY, W1, W2, F1, fscale, dF1b, dHb)
    assert bsplits == splits
    torch.cuda.synchronize()
    dF1, dH = dF1b[:M], dHb[:M]
    dYd = dY.double()
    dF1_ref = fscale * (dYd @ W2d.t()) * (F1k > 0).double()
    dF1_scale = fscale * (dYd.abs() @ W2d.abs().t())
    _row_check("dF1", dt, dF1, dF1_ref, dF1_scale, u + FP32_SLACK, _tiny(dt))
    dF1k = dF1.double()
    dH_ref = dH0.double() + dF1k @ W1d.t()
    _row_check("dH", dt, dH, dH_ref, dF1k.abs() @ W1d.abs().t() + dH0.double().abs(), FP32_SLACK)
    assert bool((dHb[M:] == SENTINEL).all()) and bool((dF1b[M:] == SENTINEL).all()), "rows >= M written"

    # ---- deterministic tickets: bit-identical repeats, self-resetting tickets, same values up to fp32 reordering ----
    if splits > 1 and ffn == 2048 and dt == "bf16":
        tickets = torch.zeros((M + 127) // 128, dtype=torch.int32, device=dev)
        outs = []
        for _ in range(2):
            xo = resid.clone()
            dh = dH0.clone()
            F1t = torch.empty(M, ffn, dtype=tdt, device=dev)
            dF1t = torch.empty(M, ffn, dtype=tdt, device=dev)
            L.ffn_fwd(X, W1, b1, W2, b2, F1t, xo, drop_ffn_p=p, ffn_bits=fbits, drop_post_p=p, post_bits=pbits, tickets=tickets)
            assert int(tickets.abs().sum()) == 0, "forward left its tickets non-zero"
            L.ffn_bwd(dY, W1, W2, F1t, fscale, dF1t, dh, tickets=tickets)
            assert int(tickets.abs().sum()) == 0, "backward left its tickets non-zero"
            outs.append((xo, dh))
        assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
        _row_check("x_out_det", dt, outs[0][0], x_out.double(), x_scale, FP32_SLACK)
        _row_check("dH_det", dt, outs[0][1], dH.double(), dF1k.abs() @ W1d.abs().t() + dH0.double().abs(), FP32_SLACK)


def test_fused_ffn_reached_every_slice_count():
    """Runs after the shape sweep: the sweep must have exercised one slice, 2, 4 and the full chunk count."""
    if not SPLITS_SEEN:
        pytest.skip("run together with test_fused_ffn_matches_fp64")
    counts = {s for s, _ in SPLITS_SEEN}
    assert {1, 2, 4} <= counts, SPLITS_SEEN
    assert any(s == c and c > 1 for s, c in SPLITS_SEEN), SPLITS_SEEN


def test_fused_ffn_refuses_bad_arguments():
    dev = "cuda"
    X = torch.zeros(128, 128, dtype=torch.bfloat16, device=dev)
    W = torch.zeros(128, 128, dtype=torch.bfloat16, device=dev)
    F1 = torch.zeros(128, 128, dtype=torch.bfloat16, device=dev)
    xo = torch.zeros(128, 128, device=dev)
    with pytest.raises(L.B200STError, match="keep bitmap"):
        L.ffn_fwd(X, W, None, W, None, F1, xo, drop_ffn_p=0.1)
    with pytest.raises(L.B200STError, match="keep bitmap"):
        L.ffn_fwd(X, W, None, W, None, F1, xo, drop_post_p=0.1)
    with pytest.raises(L.B200STError, match="fused FFN"):      # d = 192
        Xo = torch.zeros(128, 192, dtype=torch.bfloat16, device=dev)
        L.ffn_fwd(Xo, torch.zeros(192, 128, dtype=torch.bfloat16, device=dev), None,
                  torch.zeros(128, 192, dtype=torch.bfloat16, device=dev), None, F1, torch.zeros(128, 192, device=dev))
    with pytest.raises(L.B200STError, match="fused FFN"):
        L.ffn_fwd(X.float(), W.float(), None, W.float(), None, F1.float(), xo)
    with pytest.raises(L.B200STError, match="null"):
        L.check(L.load().b200st_ffn_bwd(L.BF16, None, 128, 128, 128, W.data_ptr(), W.data_ptr(), F1.data_ptr(), 1.0,
                                        F1.data_ptr(), xo.data_ptr(), None, None, L._stream()))
