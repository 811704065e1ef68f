"""The kernels at their edge shapes, element by element against fp64 references.

Every reference is computed in float64 from the same bf16- or fp32-rounded inputs the kernel reads.  Every bound is
elementwise: the output dtype's rounding (half an ulp, ``u * |ref|``) plus a term for the fp32 arithmetic before it, sized
by the longest sequential accumulation chain the kernel runs.  A failure names the worst element (largest error over
bound) by row / column, or by (batch, head, 128-row block) for attention.

The GPU tests need a B200.  The ``test_tolerance_*`` tests at the end run on the CPU: they feed each bound the fp64
reference itself, rounded to the kernel's output dtype (must pass), and deliberately wrong outputs (must fail).
"""
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tiny_deepspeed_b200 import ops

gpu = pytest.mark.gpu

U8 = 2.0 ** -8              # bf16 unit roundoff: half an ulp, relative (8 significant bits)
U24 = 2.0 ** -24            # fp32 unit roundoff
TANH_ERR = 2.0 ** -10       # tanh.approx.f32 (GELU): max relative error 2^-10.987 (PTX ISA), rounded up
FTZ = 2.0 ** -126           # smallest normal fp32 / bf16: built with --use_fast_math, results below it flush to zero
BF16, F32 = torch.bfloat16, torch.float32
LOG2E = 1.0 / math.log(2.0)


def _u(dtype):
    return U8 if dtype == BF16 else U24


def _dev():
    return torch.device("cuda", 0)


# ---------------------------------------------------------------------------------------------------------------------
# comparison
# ---------------------------------------------------------------------------------------------------------------------
def _rows_cols(idx):
    if len(idx) == 0:
        return "the scalar"
    if len(idx) == 1:
        return f"index {idx[0]}"
    return "row " + ", ".join(str(i) for i in idx[:-1]) + f" col {idx[-1]}"


def check(got, ref, bound, what, where=_rows_cols):
    """|got - ref| <= bound + FTZ elementwise (fp64; NaN fails).  On failure, name the worst element via ``where(index)``."""
    g = got.detach().double()
    r = ref.detach().double().to(g.device)
    b = torch.as_tensor(bound, dtype=torch.float64, device=g.device).expand_as(r) + FTZ
    assert g.shape == r.shape, (what, g.shape, r.shape)
    err = (g - r).abs()
    bad = ~(err <= b)
    if bool(bad.any()):
        ratio = torch.where(bad, torch.nan_to_num(err / b, nan=math.inf, posinf=math.inf), torch.zeros_like(err))
        ratio = torch.nan_to_num(ratio, nan=math.inf)
        flat = int(torch.argmax(ratio.flatten()))
        idx = tuple(int(i) for i in np.unravel_index(flat, tuple(r.shape)))
        raise AssertionError(f"{what}: {int(bad.sum())} of {r.numel()} elements out of bound; worst at {where(idx)}: "
                             f"got {g[idx].item():.8g}, want {r[idx].item():.8g}, bound {b[idx].item():.3g}")


def _attn_where(nh, packed, hs=64):
    """Index of a [B, T, nh * hs] attention tensor (or [B, T, 3 * nh * hs] when ``packed``: q, k, v) -> batch, head and
    128-row block."""
    def where(idx):
        b, t, c = idx
        part, c = divmod(c, nh * hs)
        name = "qkv"[part] if packed else ""
        return f"b={b} {name}head={c // hs} rows {t // 128 * 128}..{t // 128 * 128 + 127}"
    return where


# ---------------------------------------------------------------------------------------------------------------------
# fp64 references and their bounds (device-agnostic: the CPU tests below run the same functions)
# ---------------------------------------------------------------------------------------------------------------------
def ln_fwd_ref(x, w, b, eps, dtype):
    """(y, mean, rstd) and their bounds.  Kernel: one warp per row, fp32 two-pass mean / variance, rsqrt."""
    xd, wd, bd = x.double(), w.double(), b.double()
    N = xd.shape[1]
    mu = xd.mean(1)
    rs = (((xd - mu[:, None]) ** 2).mean(1) + eps).rsqrt()
    xh = (xd - mu[:, None]) * rs[:, None]
    y = xh * wd + bd
    chain = N / 32 + 16                                   # per-lane loop over N/32 elements + 5 shuffle levels, padded
    e_mu = chain * U24 * xd.abs().mean(1)                 # fp32 row sum
    e_rs = (2 * chain + 8) * U24                          # relative: variance sum, d = x - mu, rsqrt
    y_b = (_u(dtype) * y.abs() + wd.abs() * (rs[:, None] * e_mu[:, None] + xh.abs() * e_rs)
           + 4 * U24 * ((xh * wd).abs() + bd.abs()))      # rounding of y + error of mu and rstd + the affine's fp32 ops
    return (y, mu, rs), (y_b, e_mu + U24 * mu.abs(), e_rs * rs)


def ln_bwd_ref(dy, x, w, mean, rstd, dtype, add=None, dw0=None, db0=None):
    """(dx, dw, db) and bounds, from the fp32 mean / rstd the kernel is given.  dw0 / db0: accumulate into these."""
    dyd, xd, wd = dy.double(), x.double(), w.double()
    M, N = xd.shape
    rs = rstd.double()[:, None]
    xh = (xd - mean.double()[:, None]) * rs
    wdy = wd * dyd
    c1 = (xh * wdy).mean(1, keepdim=True)
    c2 = wdy.mean(1, keepdim=True)
    dx = (wdy - (xh * c1 + c2)) * rs
    chain = N / 32 + 20                                   # row sums of one warp, plus xhat's own fp32 rounding
    e_c1 = chain * U24 * (xh * wdy).abs().mean(1, keepdim=True)
    e_c2 = chain * U24 * wdy.abs().mean(1, keepdim=True)
    dx_b = rs * (xh.abs() * e_c1 + e_c2 + 6 * U24 * (wdy.abs() + (xh * c1).abs() + c2.abs()))
    if add is not None:
        dx = dx + add.double()
        dx_b = dx_b + U24 * add.double().abs()
    dx_b = dx_b + _u(dtype) * dx.abs()
    chain_m = M / 256 + 148 + 40                          # rows per warp, warps per CTA, then up to 148 CTA partials
    dw, db = (dyd * xh).sum(0), dyd.sum(0)
    dw_b, db_b = chain_m * U24 * (dyd * xh).abs().sum(0), chain_m * U24 * dyd.abs().sum(0)
    if dw0 is not None:
        dw, db = dw + dw0.double(), db + db0.double()
        dw_b, db_b = dw_b + U24 * dw0.double().abs(), db_b + U24 * db0.double().abs()
    return (dx, dw, db), (dx_b, dw_b + _u(dtype) * dw.abs(), db_b + _u(dtype) * db.abs())


def emb_bwd_ref(idx, dy, V, dtype, padding_idx=-1, out0=None):
    """Scatter-add reference and bound.  Atomics run in any order and round after every add, in the output dtype:
    |error| <= sum over adds of u * |partial sum| <= (count + 1) * u * (sum |dy| + |out0|) per element."""
    D = dy.shape[1]
    keep = (idx >= 0) & (idx < V) & (idx != padding_idx)
    ii, dd = idx[keep], dy.double()[keep]
    ref = torch.zeros(V, D, dtype=torch.float64, device=dy.device).index_add_(0, ii, dd)
    mag = torch.zeros(V, D, dtype=torch.float64, device=dy.device).index_add_(0, ii, dd.abs())
    cnt = torch.zeros(V, dtype=torch.float64, device=dy.device).index_add_(0, ii, torch.ones_like(ii, dtype=torch.float64))
    if out0 is not None:
        ref, mag = ref + out0.double(), mag + out0.double().abs()
    return ref, (cnt[:, None] + 1) * _u(dtype) * mag


def xent_ref(logits, tgt):
    """(loss, lse) and bounds.  Kernel: one 512-thread CTA per row, online max / sum with __expf, __logf."""
    l = logits.double()
    M, V = l.shape
    lse = torch.logsumexp(l, 1)
    p = torch.exp(l - lse[:, None])
    chain = V / 512 + 64                                  # per-thread chain (with its rescales) + block reduction
    # __expf(v - mx): argument rounding and ex2.approx, relative (|v - mx| + 4) * 2 u; weighted by each term's share
    lse_b = chain * U24 + (p * ((l - l.max(1, keepdim=True).values).abs() + 4)).sum(1) * 2 * U24 + 4 * U24 * lse.abs()
    loss = (lse - l.gather(1, tgt[:, None]).squeeze(1)).mean()
    loss_b = (lse_b + 2 * U24 * l.gather(1, tgt[:, None]).squeeze(1).abs()).mean() + (M + 4) * U24 * loss.abs()
    return (loss, lse), (loss_b, lse_b)


def xent_bwd_ref(logits, tgt, lse, gscale, dtype):
    """dlogits = (exp(l - lse) - onehot) * g / M from the fp32 lse the kernel is given; bound: __expf of a rounded
    fp32 argument (relative (2 |l - lse| + 4) u), the scaling, and the output rounding."""
    l = logits.double()
    M, V = l.shape
    z = lse.double()[:, None]
    p = torch.exp(l - z)
    oh = torch.zeros_like(p).scatter_(1, tgt[:, None], 1.0)
    g = gscale / M
    d = (p - oh) * g
    b = p * (4 * (l - z).abs() + 8) * U24 * abs(g) + 4 * U24 * d.abs() + _u(dtype) * d.abs()
    return d, b


def softmax_ref(S, scale):
    """Causal softmax of [n, T, T] scores (valid prefix [0, r] of row r) and bound.  Kernel: exp2 of the rounded fp32
    argument S * scale * log2e - max, fp32 row sum over r + 1 terms, bf16 result."""
    n, T, _ = S.shape
    mask = torch.ones(T, T, dtype=torch.bool, device=S.device).tril()
    s = (S.double() * scale).masked_fill(~mask, -math.inf)
    P = torch.softmax(s, -1)
    sf = s.masked_fill(~mask, 0.0)
    m = sf.max(-1, keepdim=True).values
    e_arg = 2 * U24 * (sf.abs() + m.abs()) + 4 * U24       # exp2 argument rounding + ex2.approx, relative to the term
    chain = (torch.arange(T, device=S.device, dtype=torch.float64) / 32 + 16)[:, None]
    rel = 2 * (e_arg + (P * e_arg).sum(-1, keepdim=True) + chain * U24)
    return P, U8 * P + P * rel


def softmax_bwd_ref(P, dP, scale):
    """dS = P * (dP - sum_j P_j dP_j) * scale over the valid prefix; fp32 dot over r + 1 terms, bf16 result."""
    n, T, _ = P.shape
    mask = torch.ones(T, T, dtype=torch.bool, device=P.device).tril()
    Pd, dPd = P.double() * mask, dP.double() * mask
    dot = (Pd * dPd).sum(-1, keepdim=True)
    dS = Pd * (dPd - dot) * scale
    chain = (torch.arange(T, device=P.device, dtype=torch.float64) / 32 + 16)[:, None]
    e_dot = chain * U24 * (Pd * dPd).abs().sum(-1, keepdim=True)
    return dS, U8 * dS.abs() + abs(scale) * Pd * (e_dot + 4 * U24 * (dPd.abs() + dot.abs()))


def attention_ref(qkv, dy, nh, y_given=None, scores_bf16=False):
    """Causal attention forward + backward in fp64 on packed qkv [B, T, 3C] (head size 64), with elementwise bounds.

    Error model (all relative errors doubled for safety): the probabilities reach the P.V / P^T.dY products as bf16
    (u8 * P; with ``scores_bf16`` the scores themselves are bf16 first, the materialised path), dP = dY.V^T and dS are
    rounded to bf16 as well, D_i = dO_i . O_i uses the bf16 forward output; every result is rounded to bf16 at the end.
    Returns dict with y, lse2 (log2 domain), dqkv and their bounds."""
    B, T, C3 = qkv.shape
    C = C3 // 3
    hs = C // nh
    scale = 1.0 / math.sqrt(hs)
    qd = qkv.double().view(B, T, 3, nh, hs).permute(2, 0, 3, 1, 4)          # [3, B, nh, T, hs]
    q, k, v = qd[0], qd[1], qd[2]
    dyd = dy.double().view(B, T, nh, hs).transpose(1, 2)
    mask = torch.ones(T, T, dtype=torch.bool, device=qkv.device).tril()
    S = q @ k.transpose(-1, -2)
    s = (S * scale).masked_fill(~mask, -math.inf)
    lse = torch.logsumexp(s, -1)
    P = torch.exp(s - lse[..., None])
    y = P @ v
    e_s = 2 * hs * U24 * (q.abs() @ k.abs().transpose(-1, -2)) * scale     # fp32 QK^T (products exact, sum of 64)
    sf = (S * scale).masked_fill(~mask, 0.0)
    e_s = e_s + 2 * U24 * (sf.abs() + sf.max(-1, keepdim=True).values.abs()) + 4 * U24   # exp2 argument, ex2.approx
    if scores_bf16:
        e_s = e_s + U8 * S.abs() * scale
    e_s = e_s.masked_fill(~mask, 0.0)
    eP = P * (2 * U8 + e_s + (P * e_s).sum(-1, keepdim=True))
    y_b = U8 * y.abs() + 2 * (eP @ v.abs())
    lse_b = (2 * (T + 64) * U24 + (P * e_s).sum(-1)) * LOG2E + 8 * U24 * lse.abs() * LOG2E
    O = y if y_given is None else y_given.double().view(B, T, nh, hs).transpose(1, 2)
    dP = dyd @ v.transpose(-1, -2)
    D = (dyd * O).sum(-1, keepdim=True)
    dS = (P * (dP - D)).masked_fill(~mask, 0.0)
    dV = P.transpose(-1, -2) @ dyd
    dQ = scale * (dS @ k)
    dK = scale * (dS.transpose(-1, -2) @ q)
    e_dP = (U8 * dP.abs()).masked_fill(~mask, 0.0)
    eD = (2 * U8 * (dyd.abs() * O.abs()).sum(-1, keepdim=True) + (eP * dP.abs()).sum(-1, keepdim=True)
          + (P * e_dP).sum(-1, keepdim=True))
    edS = (U8 * dS.abs() + eP * (dP - D).abs() + P * (e_dP + eD)).masked_fill(~mask, 0.0)
    dV_b = U8 * dV.abs() + 2 * (eP.transpose(-1, -2) @ dyd.abs())
    dQ_b = U8 * dQ.abs() + 2 * scale * (edS @ k.abs())
    dK_b = U8 * dK.abs() + 2 * scale * (edS.transpose(-1, -2) @ q.abs())

    def pack(t):                                                             # [B, nh, T, hs] -> [B, T, C]
        return t.transpose(1, 2).reshape(B, T, C)
    return dict(y=pack(y), y_b=pack(y_b), lse2=lse * LOG2E, lse2_b=lse_b,
                dqkv=torch.cat([pack(dQ), pack(dK), pack(dV)], 2), dqkv_b=torch.cat([pack(dQ_b), pack(dK_b), pack(dV_b)], 2))


def gemm_acc_bound(a, b, alpha=1.0):
    """fp32 tensor-core accumulation over K of exact bf16 products: <= 2 K u32 sum_k |a||b| (rounding or truncation)."""
    K = a.shape[1]
    return 2 * K * U24 * abs(alpha) * (a.double().abs() @ b.double().abs().t())


def gelu_ref(x):
    k0, k1 = 0.7978845608028654, 0.044715
    xd = x.double()
    t = torch.tanh(k0 * (xd + k1 * xd ** 3))
    return 0.5 * xd * (1 + t), 0.5 * xd.abs() * t.abs() * TANH_ERR + 4 * U24 * xd.abs()


def gelu_grad_ref(x):
    k0, k1 = 0.7978845608028654, 0.044715
    xd = x.double()
    t = torch.tanh(k0 * (xd + k1 * xd ** 3))
    g = 0.5 * (1 + t) + 0.5 * xd * (1 - t * t) * k0 * (1 + 3 * k1 * xd * xd)
    # d g / d t = 0.5 - x t k0 (1 + 3 k1 x^2), times the tanh.approx error; plus the fp32 arithmetic
    return g, t.abs() * TANH_ERR * (0.5 + xd.abs() * t.abs() * k0 * (1 + 3 * k1 * xd * xd)) + 8 * U24 * (g.abs() + 1)


def colsum_ref(x, dtype, out0=None):
    """Column sums; kernel: 8 row-lanes striding M, then an 8-way fold, in fp32."""
    xd = x.double()
    M = xd.shape[0]
    ref = xd.sum(0)
    b = (M / 8 + 16) * U24 * xd.abs().sum(0)
    if out0 is not None:
        ref, b = ref + out0.double(), b + U24 * out0.double().abs()
    return ref, b + _u(dtype) * ref.abs()


# ---------------------------------------------------------------------------------------------------------------------
# LayerNorm
# ---------------------------------------------------------------------------------------------------------------------
LN_N = [1, 7, 100, 200, 769, 1600, 2048, 2056, 3072]
LN_M = [1, 3, 1024, 4099]


def _ln_inputs(M, N, dtype, seed, mean=0.0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = (mean + torch.randn(M, N, device=_dev(), generator=g)).to(dtype)
    w = (torch.rand(N, device=_dev(), generator=g) + 0.5).to(dtype)
    b = torch.randn(N, device=_dev(), generator=g).to(dtype)
    dy = torch.randn(M, N, device=_dev(), generator=g).to(dtype)
    add = torch.randn(M, N, device=_dev(), generator=g).to(dtype)
    return x, w, b, dy, add


def _ln_case(x, w, b, dy, add, dtype, variants, tag):
    M, N = x.shape
    (y_r, mu_r, rs_r), (y_b, mu_b, rs_b) = ln_fwd_ref(x, w, b, 1e-5, dtype)
    y, mean, rstd = ops.layernorm_fwd(x, w, b, 1e-5)
    check(y, y_r, y_b, f"{tag} y")
    check(mean, mu_r, mu_b, f"{tag} mean")
    check(rstd, rs_r, rs_b, f"{tag} rstd")
    # backward from the kernel's own statistics (the fp32 values it is handed); dw / db accumulate into non-zero buffers
    dw0 = torch.randn(N, device=_dev()).to(dtype)
    db0 = torch.randn(N, device=_dev()).to(dtype)
    (dx_r, dw_r, db_r), (dx_b, dw_b, db_b) = ln_bwd_ref(dy, x, w, mean, rstd, dtype, add=add)
    (_, dwa_r, dba_r), (_, dwa_b, dba_b) = ln_bwd_ref(dy, x, w, mean, rstd, dtype, dw0=dw0, db0=db0)
    for variant in variants:
        dw, db = torch.empty_like(w), torch.empty_like(w)
        dx = ops.ext().layernorm_bwd(dy, x, w, mean, rstd, dw, db, False, add, variant)
        check(dx, dx_r, dx_b, f"{tag} variant {variant} dx (add_to_dx)")
        check(dw, dw_r, dw_b, f"{tag} variant {variant} dw")
        check(db, db_r, db_b, f"{tag} variant {variant} db")
        dw, db = dw0.clone(), db0.clone()
        ops.ext().layernorm_bwd(dy, x, w, mean, rstd, dw, db, True, None, variant)
        check(dw, dwa_r, dwa_b, f"{tag} variant {variant} dw (accumulate)")
        check(db, dba_r, dba_b, f"{tag} variant {variant} db (accumulate)")


@gpu
@pytest.mark.parametrize("M", LN_M)
@pytest.mark.parametrize("dtype", [BF16, F32], ids=["bf16", "fp32"])
@pytest.mark.parametrize("N", LN_N)
def test_layernorm_edges(N, dtype, M):
    """Every width (vector path, scalar tail, scalar-only rows), both dtypes, both backward arms; bf16 at N % 8 == 0 and
    N <= 2048 runs the register-resident backward in both its forms (variant 0: partials + fold, 1: single launch)."""
    x, w, b, dy, add = _ln_inputs(M, N, dtype, seed=N * 10 + M)
    fast = dtype == BF16 and N % 8 == 0 and N <= 2048
    _ln_case(x, w, b, dy, add, dtype, (0, 1) if fast else (-1,), f"N={N} M={M}")


@gpu
@pytest.mark.parametrize("dtype", [BF16, F32], ids=["bf16", "fp32"])
@pytest.mark.parametrize("N", [7, 768, 3072])
def test_layernorm_large_mean(N, dtype):
    """x = 50 + randn: a one-pass E[x^2] - E[x]^2 variance would cancel to garbage; the bound leaves no room for that."""
    x, w, b, dy, add = _ln_inputs(1024, N, dtype, seed=N, mean=50.0)
    _ln_case(x, w, b, dy, add, dtype, (0, 1) if dtype == BF16 and N % 8 == 0 else (-1,), f"mean 50 N={N}")


@gpu
def test_layernorm_single_launch_accumulators_clean_across_widths():
    """The single-launch backward keeps persistent fp32 accumulators laid out by N; 768 -> 1600 -> 768 shows the last
    CTA leaves them zeroed whatever width came before."""
    for i, N in enumerate((768, 1600, 768)):
        x, w, b, dy, _ = _ln_inputs(1024, N, BF16, seed=100 + i)
        _, mean, rstd = ops.layernorm_fwd(x, w, b, 1e-5)
        (dx_r, dw_r, db_r), (dx_b, dw_b, db_b) = ln_bwd_ref(dy, x, w, mean, rstd, BF16)
        dw, db = torch.empty_like(w), torch.empty_like(w)
        dx = ops.ext().layernorm_bwd(dy, x, w, mean, rstd, dw, db, False, None, 1)
        check(dx, dx_r, dx_b, f"pass {i} N={N} dx")
        check(dw, dw_r, dw_b, f"pass {i} N={N} dw")
        check(db, db_r, db_b, f"pass {i} N={N} db")


# ---------------------------------------------------------------------------------------------------------------------
# Embedding
# ---------------------------------------------------------------------------------------------------------------------
EMB_DIMS = [1, 3, 64, 100, 768, 770]


@gpu
@pytest.mark.parametrize("dtype", [BF16, F32], ids=["bf16", "fp32"])
@pytest.mark.parametrize("dim", EMB_DIMS)
def test_embedding_edges(dim, dtype):
    V, ntok, add_rows, pad = 97, 600, 37, 5
    g = torch.Generator(device="cuda").manual_seed(dim)
    w = torch.randn(V, dim, device=_dev(), generator=g).to(dtype)
    idx = torch.randint(0, V, (ntok,), device=_dev(), generator=g)
    idx[:9] = pad
    pos = torch.randn(add_rows, dim, device=_dev(), generator=g).to(dtype)
    # forward: plain gather is exact; with `add` (row tok % add_rows, add_rows < ntok) one fp32 add, then the rounding
    out = ops.embedding_forward(idx, w)
    check(out, w.double()[idx], 0.0, f"dim={dim} gather")
    out = ops.embedding_forward(idx, w, add=pos)
    ref = w.double()[idx] + pos.double()[torch.arange(ntok, device=_dev()) % add_rows]
    check(out, ref, _u(dtype) * ref.abs(), f"dim={dim} gather + add")
    # backward: padding_idx rows get nothing; accumulate=True adds into a non-zero gradient
    dy = torch.randn(ntok, dim, device=_dev(), generator=g).to(dtype)
    gw = ops.embedding_weight_grad(idx, dy, w, padding_idx=pad)
    ref, bound = emb_bwd_ref(idx, dy, V, dtype, padding_idx=pad)
    check(gw, ref, bound, f"dim={dim} scatter-add")
    assert torch.all(gw[pad] == 0)
    out0 = torch.randn(V, dim, device=_dev(), generator=g).to(dtype)
    acc = out0.clone()
    ops.embedding_weight_grad(idx, dy, w, out=acc, accumulate=True)
    ref, bound = emb_bwd_ref(idx, dy, V, dtype, out0=out0)
    check(acc, ref, bound, f"dim={dim} scatter-add (accumulate)")


@gpu
@pytest.mark.parametrize("dtype", [BF16, F32], ids=["bf16", "fp32"])
@pytest.mark.parametrize("dim", [3, 770])
def test_embedding_one_id_repeated_4096_times(dim, dtype):
    """4096 atomics onto one row.  The values are chosen so that no add can round: fp32 gets k/16 for |k| <= 8 (every
    partial sum is a multiple of 1/16 below 2^11, 15 bits); bf16 gets +-1/8 in 256 of the 4096 rows of each column
    (every partial sum is a multiple of 1/8 of magnitude <= 32, 8 bits).  Per-add rounding is then zero in any order,
    so the result must be exact."""
    ntok, V = 4096, 11
    g = torch.Generator(device="cuda").manual_seed(dim)
    idx = torch.full((ntok,), 7, dtype=torch.long, device=_dev())
    if dtype == F32:
        dy = torch.randint(-8, 9, (ntok, dim), device=_dev(), generator=g).float() / 16
    else:
        sign = torch.randint(0, 2, (ntok, dim), device=_dev(), generator=g) * 2 - 1
        t = torch.arange(ntok, device=_dev())[:, None] + torch.arange(dim, device=_dev())[None]
        dy = (sign * (t % 16 == 0) / 8.0).to(BF16)
    gw = ops.embedding_weight_grad(idx, dy, torch.empty(V, dim, device=_dev(), dtype=dtype))
    ref, _ = emb_bwd_ref(idx, dy, V, dtype)
    check(gw, ref, 0.0, f"dim={dim} repeated id")


# ---------------------------------------------------------------------------------------------------------------------
# Cross-entropy
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("scale", [1.0, 30.0])
@pytest.mark.parametrize("M", [1, 7, 1024])
@pytest.mark.parametrize("dtype", [BF16, F32], ids=["bf16", "fp32"])
@pytest.mark.parametrize("V", [8, 1000, 1001, 50257, 50304])
def test_cross_entropy_edges(V, dtype, M, scale):
    g = torch.Generator(device="cuda").manual_seed(V + M)
    l = torch.randn(M, V, device=_dev(), generator=g) * scale
    t = torch.randint(0, V, (M,), device=_dev(), generator=g)
    if M > 1:
        l[1] = 0.25                                   # all-equal row: lse = 0.25 + ln V
    l[0, t[0]] = l[0].max() + 200.0                   # one dominating logit: row loss ~ 0
    l = l.to(dtype)
    loss, lse = ops.cross_entropy_forward(l, t)
    (loss_r, lse_r), (loss_b, lse_b) = xent_ref(l, t)
    check(lse, lse_r, lse_b, f"V={V} M={M} lse")
    check(loss, loss_r, loss_b, f"V={V} M={M} loss")
    if M > 1:
        assert abs(lse[1].item() - (0.25 + math.log(V))) <= lse_b[1].item() + 1e-6
    gl = 0.37
    d = ops.cross_entropy_backward(torch.tensor(gl, device=_dev()), l, t, lse)
    d_r, d_b = xent_bwd_ref(l, t, lse, gl, dtype)
    check(d, d_r, d_b, f"V={V} M={M} dlogits")


# ---------------------------------------------------------------------------------------------------------------------
# Causal softmax (materialised-score attention): fast kernel T <= 1024, T <= 2048, generic kernel above
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("T,nmat", [(8, 3), (136, 2), (1024, 1), (1032, 2), (2048, 1), (2056, 2), (4096, 3)])
def test_causal_softmax_edges(T, nmat):
    g = torch.Generator(device="cuda").manual_seed(T)
    mask = torch.ones(T, T, dtype=torch.bool, device=_dev()).tril()
    scale = 0.125
    S = (torch.randn(nmat, T, T, device=_dev(), generator=g) * 16).masked_fill(~mask, 1e4).to(BF16)   # junk above
    P_r, P_b = softmax_ref(S, scale)
    P = S.clone()
    ops.ext().softmax_causal_fwd(P, scale)
    check(P, P_r, P_b, f"T={T} softmax P", where=lambda i: f"matrix {i[0]} row {i[1]} col {i[2]}")
    assert torch.all(P.masked_select(~mask) == 0), "masked suffix of P must be exactly zero"
    dP = torch.randn(nmat, T, T, device=_dev(), generator=g).masked_fill(~mask, 1e4).to(BF16)
    dS_r, dS_b = softmax_bwd_ref(P, dP, scale)
    dS = dP.clone()
    ops.ext().softmax_causal_bwd(P, dS, scale)
    check(dS, dS_r, dS_b, f"T={T} softmax dS", where=lambda i: f"matrix {i[0]} row {i[1]} col {i[2]}")
    assert torch.all(dS.masked_select(~mask) == 0), "masked suffix of dS must be exactly zero"


# ---------------------------------------------------------------------------------------------------------------------
# GEMM with a bf16 output whose N or row pitch is not a multiple of 8 (direct epilogue, scalar tail)
# ---------------------------------------------------------------------------------------------------------------------
def _out_view(M, N, pad):
    return torch.empty(M, N + pad, device=_dev(), dtype=BF16)[:, :N]


@gpu
@pytest.mark.parametrize("M", [1, 129, 1024])
@pytest.mark.parametrize("N,pad", [(1, 0), (100, 0), (1001, 0), (96, 3)])
def test_gemm_bf16_unaligned_epilogues(N, pad, M):
    K = 256
    g = torch.Generator(device="cuda").manual_seed(N + M)
    a = torch.randn(M, K, device=_dev(), generator=g).to(BF16)
    b = (torch.randn(N, K, device=_dev(), generator=g) * 0.1).to(BF16)
    bias = torch.randn(N, device=_dev(), generator=g).to(BF16)
    acc = a.double() @ b.double().t()
    e_acc = gemm_acc_bound(a, b)
    where = _rows_cols

    out = _out_view(M, N, pad)
    ops.gemm(a, b, out=out)
    check(out, acc, U8 * acc.abs() + e_acc, f"M={M} N={N} ldd={N + pad} no epilogue", where)

    out = _out_view(M, N, pad)
    ops.gemm(a, b, out=out, bias=bias)
    ref = acc + bias.double()
    check(out, ref, U8 * ref.abs() + e_acc + 2 * U24 * ref.abs(), f"M={M} N={N} bias", where)

    pre = _out_view(M, N, pad + 5)
    out = _out_view(M, N, pad)
    ops.gemm(a, b, out=out, bias=bias, aux=pre, epi=ops.EPI_GELU_SAVE)
    check(pre, ref, U8 * ref.abs() + e_acc + 2 * U24 * ref.abs(), f"M={M} N={N} GELU_SAVE pre-activation", where)
    gr, gb = gelu_ref(pre)                            # the epilogue applies GELU to the bf16 pre-activation it stored
    check(out, gr, U8 * gr.abs() + gb, f"M={M} N={N} GELU_SAVE output", where)

    aux = (torch.randn(M, N, device=_dev(), generator=g) * 3).to(BF16)
    out = _out_view(M, N, pad)
    ops.gemm(a, b, out=out, aux=aux, epi=ops.EPI_GELU_BWD)
    gd, gdb = gelu_grad_ref(aux)
    ref = acc * gd
    check(out, ref, U8 * ref.abs() + e_acc * gd.abs() + acc.abs() * gdb, f"M={M} N={N} GELU_BWD", where)

    out = _out_view(M, N, pad)
    ops.gemm(a, b, out=out, bias=bias, aux=aux, epi=ops.EPI_RESIDUAL)
    ref = acc + bias.double() + aux.double()
    check(out, ref, U8 * ref.abs() + e_acc + 4 * U24 * ref.abs(), f"M={M} N={N} RESIDUAL", where)

    base = torch.randn(M, N + pad, device=_dev(), generator=g).to(BF16)
    pad_before = base[:, N:].clone()
    out = base[:, :N]
    out0 = out.double().clone()
    ops.gemm(a, b, out=out, accumulate=True, alpha=-0.75)
    ref = out0 - 0.75 * acc
    check(out, ref, U8 * ref.abs() + 0.75 * e_acc + 4 * U24 * ref.abs(), f"M={M} N={N} accumulate alpha", where)
    assert torch.equal(base[:, N:], pad_before), "the epilogue wrote past column N of the output view"


@gpu
def test_lm_head_forward_vocab_50257():
    """The real GPT-2 vocabulary: [1024, 768] x [50257, 768]^T; the logits rows are 100514 bytes apart."""
    g = torch.Generator(device="cuda").manual_seed(50257)
    x = torch.randn(1024, 768, device=_dev(), generator=g).to(BF16)
    w = (torch.randn(50257, 768, device=_dev(), generator=g) * 0.05).to(BF16)
    y = ops.linear_forward(x, w)
    acc = x.double() @ w.double().t()
    check(y, acc, U8 * acc.abs() + gemm_acc_bound(x, w), "lm_head logits")
    t = torch.randint(0, 50257, (1024,), device=_dev(), generator=g)
    loss, lse = ops.cross_entropy_forward(y, t)
    (loss_r, lse_r), (loss_b, lse_b) = xent_ref(y, t)
    check(lse, lse_r, lse_b, "lm_head lse")
    check(loss, loss_r, loss_b, "lm_head loss")


# ---------------------------------------------------------------------------------------------------------------------
# Flash attention (head size 64, T % 128 == 0) and the materialised fallback (T = 136)
# ---------------------------------------------------------------------------------------------------------------------
def _attn_inputs(B, T, nh, scale, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    C = nh * 64
    qkv = (torch.randn(B, T, 3 * C, device=_dev(), generator=g) * scale).to(BF16)
    dy = torch.randn(B, T, C, device=_dev(), generator=g).to(BF16)
    return qkv, dy


def _check_attention(y, lse, dqkv, r, nh, tag):
    check(y, r["y"], r["y_b"], f"{tag} y", _attn_where(nh, False))
    if lse is not None:
        check(lse, r["lse2"], r["lse2_b"], f"{tag} lse (log2 domain)",
              where=lambda i: f"b={int(i[0])} head={int(i[1])} rows {int(i[2]) // 128 * 128}..")
    check(dqkv, r["dqkv"], r["dqkv_b"], f"{tag} dqkv", _attn_where(nh, True))


@gpu
@pytest.mark.parametrize("qscale", [0.7, 2.5])
@pytest.mark.parametrize("B,T,nh", [(1, 256, 2), (2, 1152, 3), (4, 512, 25), (1, 2048, 4)])
def test_flash_attention_edges(B, T, nh, qscale):
    qkv, dy = _attn_inputs(B, T, nh, qscale, seed=T + nh)
    assert ops.ext().flash_supported(T, 64)
    y, lse = ops.causal_attention_forward(qkv, nh)
    dqkv = ops.causal_attention_backward(dy, qkv, lse, nh, y=y)
    r = attention_ref(qkv, dy, nh, y_given=y)
    _check_attention(y, lse, dqkv, r, nh, f"B={B} T={T} nh={nh} scale={qscale}")
    # dK / dV of a split key block are two fp32 partials TMA-added into a workspace that flash_dsum_kernel zeroes:
    # 0 + a + b == 0 + b + a exactly, so they are bit-identical run to run (dQ is a many-way reduce-add: not compared).
    # The second call gets the first call's freed workspace back from the allocator, stale sums included.
    C = nh * 64
    again = ops.causal_attention_backward(dy, qkv, lse, nh, y=y)
    assert torch.equal(again[..., C:], dqkv[..., C:]), "dK / dV differ between two identical backward calls"


_SPLIT0_SCRIPT = r"""
import sys, torch
sys.path.insert(0, sys.argv[1])
from tiny_deepspeed_b200 import ops
d = torch.load(sys.argv[2])
qkv, dy, nh = d["qkv"].cuda(), d["dy"].cuda(), d["nh"]
y, lse = ops.causal_attention_forward(qkv, nh)
dqkv = ops.causal_attention_backward(dy, qkv, lse, nh, y=y)
torch.save({"y": y.cpu(), "lse": lse.cpu(), "dqkv": dqkv.cpu()}, sys.argv[3])
"""


@gpu
def test_flash_backward_unsplit_arm(tmp_path):
    """TDS_FLASH_SPLIT=0 (one CTA per key block) is read once per process, so it runs in a child process: its dqkv
    must meet the fp64 bound, and agree with the default (split) arm within the sum of both bounds."""
    B, T, nh = 1, 2048, 4
    qkv, dy = _attn_inputs(B, T, nh, 0.7, seed=7)
    torch.save({"qkv": qkv.cpu(), "dy": dy.cpu(), "nh": nh}, tmp_path / "in.pt")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, TDS_FLASH_SPLIT="0")
    flags = ["-s"] if sys.flags.no_user_site else []
    r = subprocess.run([sys.executable, *flags, "-c", _SPLIT0_SCRIPT, root, str(tmp_path / "in.pt"), str(tmp_path / "out.pt")],
                       env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    other = torch.load(tmp_path / "out.pt")
    y, lse = ops.causal_attention_forward(qkv, nh)
    dqkv = ops.causal_attention_backward(dy, qkv, lse, nh, y=y)
    assert torch.equal(other["y"].cuda(), y) and torch.equal(other["lse"].cuda(), lse), "forward must not depend on the split"
    ref = attention_ref(qkv, dy, nh, y_given=y)
    _check_attention(y, lse, other["dqkv"].cuda(), ref, nh, "TDS_FLASH_SPLIT=0")
    check(other["dqkv"].cuda(), dqkv, 2 * ref["dqkv_b"], "split arm vs unsplit arm", _attn_where(nh, True))


@gpu
def test_attention_materialised_fallback_t136():
    """T = 136 is not a multiple of 128: the attention runs as GEMMs over bf16 scores + the causal softmax kernels."""
    B, T, nh = 2, 136, 3
    qkv, dy = _attn_inputs(B, T, nh, 0.7, seed=136)
    assert not ops.ext().flash_supported(T, 64)
    y, P = ops.causal_attention_forward(qkv, nh)
    assert P.dtype == BF16 and P.shape == (B, nh, T, T)
    dqkv = ops.causal_attention_backward(dy, qkv, P, nh, y=y)
    r = attention_ref(qkv, dy, nh, scores_bf16=True)
    _check_attention(y, None, dqkv, r, nh, "T=136 materialised")


# ---------------------------------------------------------------------------------------------------------------------
# GELU, column sum, cast
# ---------------------------------------------------------------------------------------------------------------------
EW_N = [1, 7, 2 * 148 * 256 * 64 + 3]     # the last: more than one grid-stride pass at the 148 * 8-block cap, + a tail


@gpu
@pytest.mark.parametrize("dtype", [BF16, F32], ids=["bf16", "fp32"])
@pytest.mark.parametrize("n", EW_N)
def test_gelu_and_cast_edges(n, dtype):
    g = torch.Generator(device="cuda").manual_seed(n)
    x = ((torch.rand(n, device=_dev(), generator=g) * 2 - 1) * 12).to(dtype)
    dy = torch.randn(n, device=_dev(), generator=g).to(dtype)
    gr, gb = gelu_ref(x)
    check(ops.gelu_forward(x), gr, _u(dtype) * gr.abs() + gb, f"n={n} gelu")
    gd, gdb = gelu_grad_ref(x)
    ref = dy.double() * gd
    check(ops.gelu_backward(dy, x), ref, _u(dtype) * ref.abs() + dy.double().abs() * gdb, f"n={n} gelu'")
    other = F32 if dtype == BF16 else BF16
    c = ops.cast(x, other)
    assert c.dtype == other and torch.equal(c, x.to(other))       # bf16 -> fp32 exact, fp32 -> bf16 round-to-nearest-even


@gpu
@pytest.mark.parametrize("dtype", [BF16, F32], ids=["bf16", "fp32"])
@pytest.mark.parametrize("M,N", [(1, 1001), (1024, 1001), (4099, 33), (3, 7)])
def test_colsum_edges(M, N, dtype):
    g = torch.Generator(device="cuda").manual_seed(M * N)
    x = torch.randn(M, N, device=_dev(), generator=g).to(dtype)
    out = ops.linear_bias_grad(x)
    ref, b = colsum_ref(x, dtype)
    check(out, ref, b, f"M={M} N={N} colsum")
    out0 = torch.randn(N, device=_dev(), generator=g).to(dtype)
    acc = out0.clone()
    ops.linear_bias_grad(x, out=acc, accumulate=True)
    ref, b = colsum_ref(x, dtype, out0=out0)
    check(acc, ref, b, f"M={M} N={N} colsum (accumulate)")


# ---------------------------------------------------------------------------------------------------------------------
# Row kernels on 16-byte-misaligned views (contiguous, but starting one element into their storage)
# ---------------------------------------------------------------------------------------------------------------------
def _offset_view(t):
    buf = torch.empty(t.numel() + 1, device=t.device, dtype=t.dtype)
    v = buf[1:].view(t.shape)
    v.copy_(t)
    return v


@gpu
@pytest.mark.parametrize("dtype", [BF16, F32], ids=["bf16", "fp32"])
def test_row_kernels_on_offset_views(dtype):
    M, N = 1024, 768
    x, w, b, dy, add = _ln_inputs(M, N, dtype, seed=1)
    xo, wo, bo, dyo = (_offset_view(t) for t in (x, w, b, dy))
    assert xo.data_ptr() % 16 != 0 and xo.is_contiguous()
    _ln_case(xo, wo, bo, dyo, _offset_view(add), dtype, (0, 1) if dtype == BF16 else (-1,), "offset view")
    V = 1000
    emb = _offset_view(torch.randn(V, N, device=_dev()).to(dtype))
    idx = torch.randint(0, V, (300,), device=_dev())
    check(ops.embedding_forward(idx, emb), emb.double()[idx], 0.0, "offset view gather")
    dy2 = torch.randn(300, N, device=_dev()).to(dtype)
    gw = _offset_view(torch.zeros(V, N, device=_dev(), dtype=dtype))
    ops.embedding_weight_grad(idx, dy2, emb, out=gw, accumulate=True)
    ref, bound = emb_bwd_ref(idx, dy2, V, dtype)
    check(gw, ref, bound, "offset view scatter-add")
    l = _offset_view((torch.randn(64, 50304, device=_dev()) * 3).to(dtype))
    t = torch.randint(0, 50304, (64,), device=_dev())
    loss, lse = ops.cross_entropy_forward(l, t)
    (loss_r, lse_r), (loss_b, lse_b) = xent_ref(l, t)
    check(lse, lse_r, lse_b, "offset view lse")
    d = _offset_view(torch.empty_like(l))
    ops.cross_entropy_backward(torch.tensor(1.0, device=_dev()), l, t, lse, out=d)
    d_r, d_b = xent_bwd_ref(l, t, lse, 1.0, dtype)
    check(d, d_r, d_b, "offset view dlogits")


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the bounds pass the correctly rounded reference and fail the bugs they exist to catch
# ---------------------------------------------------------------------------------------------------------------------
def _rounded(t, dtype):
    """The fp64 reference as the kernel would store it: rounded to its output dtype."""
    return t.to(dtype).double()


@pytest.mark.parametrize("dtype", [BF16, F32], ids=["bf16", "fp32"])
def test_tolerance_layernorm_catches_neighbour_row_and_zeroed_tail(dtype):
    torch.manual_seed(0)
    M, N = 6, 7
    x = torch.randn(M, N).to(dtype)
    w = (torch.rand(N) + 0.5).to(dtype)
    b = torch.randn(N).to(dtype)
    (y, mu, rs), (y_b, mu_b, rs_b) = ln_fwd_ref(x, w, b, 1e-5, dtype)
    check(_rounded(y, dtype), y, y_b, "rounded y")
    check(mu.float(), mu, mu_b, "rounded mean")
    check(rs.float(), rs, rs_b, "rounded rstd")
    wrong = y.clone()
    wrong[3] = y[2]
    with pytest.raises(AssertionError, match="row 3"):
        check(_rounded(wrong, dtype), y, y_b, "neighbour row")
    wrong = y.clone()
    wrong[:, -1] = 0
    with pytest.raises(AssertionError, match="col 6"):
        check(_rounded(wrong, dtype), y, y_b, "zeroed tail")
    dy = torch.randn(M, N).to(dtype)
    (dx, dw, db), (dx_b, dw_b, db_b) = ln_bwd_ref(dy, x, w, mu.float(), rs.float(), dtype)
    check(_rounded(dx, dtype), dx, dx_b, "rounded dx")
    check(_rounded(dw, dtype), dw, dw_b, "rounded dw")
    wrong = dx.clone()
    wrong[1] = dx[0]
    with pytest.raises(AssertionError, match="row 1"):
        check(_rounded(wrong, dtype), dx, dx_b, "neighbour row dx")
    with pytest.raises(AssertionError):
        check(_rounded(dw - dy.double()[M - 1] * ((x.double()[M - 1] - mu[M - 1]) * rs[M - 1]), dtype), dw, dw_b,
              "dw missing the last row")


@pytest.mark.parametrize("dtype", [BF16, F32], ids=["bf16", "fp32"])
@pytest.mark.parametrize("dim", [3, 9])
def test_tolerance_embedding_catches_zeroed_last_column(dim, dtype):
    torch.manual_seed(dim)
    V, ntok = 16, 128
    idx = torch.randint(0, V, (ntok,))
    dy = torch.randn(ntok, dim).to(dtype)
    ref, bound = emb_bwd_ref(idx, dy, V, dtype)
    check(_rounded(ref, dtype), ref, bound, "rounded scatter-add")
    wrong = ref.clone()
    wrong[:, -1] = 0
    with pytest.raises(AssertionError, match=f"col {dim - 1}"):
        check(_rounded(wrong, dtype), ref, bound, "zeroed last column")


@pytest.mark.parametrize("dtype", [BF16, F32], ids=["bf16", "fp32"])
def test_tolerance_cross_entropy_catches_neighbour_row(dtype):
    torch.manual_seed(1)
    M, V = 8, 1001
    l = (torch.randn(M, V) * 3).to(dtype)
    t = torch.randint(0, V, (M,))
    (loss, lse), (loss_b, lse_b) = xent_ref(l, t)
    check(lse.float(), lse, lse_b, "rounded lse")
    check(loss.float(), loss, loss_b, "rounded loss")
    wrong = lse.clone()
    wrong[5] = lse[4]
    with pytest.raises(AssertionError, match="index 5"):
        check(wrong.float(), lse, lse_b, "neighbour lse")
    d, d_b = xent_bwd_ref(l, t, lse.float(), 0.37, dtype)
    check(_rounded(d, dtype), d, d_b, "rounded dlogits")
    wrong = d.clone()
    wrong[5] = d[4]
    with pytest.raises(AssertionError, match="row 5"):
        check(_rounded(wrong, dtype), d, d_b, "neighbour dlogits")


@pytest.mark.parametrize("dtype", [BF16, F32], ids=["bf16", "fp32"])
def test_tolerance_colsum_catches_bf16_accumulation(dtype):
    torch.manual_seed(2)
    M, N = 1024, 40
    x = torch.randn(M, N).to(dtype)
    ref, bound = colsum_ref(x, dtype)
    check(_rounded(ref, dtype), ref, bound, "rounded colsum")
    acc = torch.zeros(N, dtype=BF16)
    for r in range(M):                                # a running sum kept in bf16, as a wrong kernel would
        acc = (acc.float() + x[r].float()).to(BF16)
    with pytest.raises(AssertionError):
        check(acc, ref, bound, "bf16-accumulated colsum")


def _small_attention(B=1, T=256, nh=2, scale=0.7, seed=3):
    g = torch.Generator().manual_seed(seed)
    C = nh * 64
    qkv = (torch.randn(B, T, 3 * C, generator=g) * scale).to(BF16)
    dy = torch.randn(B, T, C, generator=g).to(BF16)
    return qkv, dy


def test_tolerance_attention_lse_is_log2_domain():
    qkv, dy = _small_attention()
    r = attention_ref(qkv, dy, 2)
    lse2 = r["lse2"]
    check(lse2.float(), lse2, r["lse2_b"], "rounded lse")
    with pytest.raises(AssertionError):
        check((lse2 * math.log(2.0)).float(), lse2, r["lse2_b"], "natural-log lse")


@pytest.mark.parametrize("scores_bf16", [False, True])
def test_tolerance_attention_catches_block_from_another_head(scores_bf16):
    nh = 2
    qkv, dy = _small_attention(nh=nh)
    r = attention_ref(qkv, dy, nh, scores_bf16=scores_bf16)
    y, dqkv = r["y"], r["dqkv"]
    check(_rounded(y, BF16), y, r["y_b"], "rounded y", _attn_where(nh, False))
    check(_rounded(dqkv, BF16), dqkv, r["dqkv_b"], "rounded dqkv", _attn_where(nh, True))
    wrong = y.clone()
    wrong[0, 128:256, 64:128] = y[0, 128:256, 0:64]  # head 1, second 128-row block <- head 0's
    with pytest.raises(AssertionError, match=r"b=0 head=1 rows 128\.\.255"):
        check(_rounded(wrong, BF16), y, r["y_b"], "y block from another head", _attn_where(nh, False))
    for part in range(3):                             # dQ, dK, dV: head 0's first block <- head 1's
        wrong = dqkv.clone()
        c0 = part * nh * 64
        wrong[0, 0:128, c0:c0 + 64] = dqkv[0, 0:128, c0 + 64:c0 + 128]
        with pytest.raises(AssertionError, match=rf"b=0 {'qkv'[part]}head=0 rows 0\.\.127"):
            check(_rounded(wrong, BF16), dqkv, r["dqkv_b"], "dqkv block from another head", _attn_where(nh, True))


def test_tolerance_softmax_and_gelu_pass_rounded_reference():
    torch.manual_seed(4)
    T = 24
    S = (torch.randn(2, T, T) * 16).to(BF16)
    P, P_b = softmax_ref(S, 0.125)
    check(_rounded(P, BF16), P, P_b, "rounded P")
    wrong = P.clone()
    wrong[1, 10] = P[1, 9]
    with pytest.raises(AssertionError, match="row 1, 10"):
        check(_rounded(wrong, BF16), P, P_b, "neighbour row P")
    dP = torch.randn(2, T, T).to(BF16)
    Pb = P.to(BF16)
    dS, dS_b = softmax_bwd_ref(Pb, dP, 0.125)
    check(_rounded(dS, BF16), dS, dS_b, "rounded dS")
    x = torch.linspace(-12, 12, 1001).to(BF16)
    gr, gb = gelu_ref(x)
    check(_rounded(gr, BF16), gr, U8 * gr.abs() + gb, "rounded gelu")
    gd, gdb = gelu_grad_ref(x)
    check(_rounded(gd, BF16), gd, U8 * gd.abs() + gdb, "rounded gelu'")
