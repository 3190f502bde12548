"""Stand-alone tests of every textual-head kernel of csrc/head.cu, and of each of its size-dispatched variants, against
fp64 references written from the textbook formulas.

The references reproduce only the kernels' documented rounding points: the bf16 input tensors; in attention the bf16
rounding of exp(s - max) * dropscale before P.V (the row sum is taken before rounding), of P * mask before dV and of dS
before dQ / dK; in GELU the bf16 rounding of gelu(u) before the dropout scale.  Everything else is fp64.  Dropout
masks come from `keep_scale`, a numpy copy of the counter-based hash of csrc/vtx_common.cuh, so every dropout case is
compared element by element.

Every comparison is made per unit (a row of a LayerNorm / cross-entropy output, a column of a column sum / dgamma, a
(batch, head) block of attention): one wrong unit fails the test.  Each check prints its worst error / tolerance ratio.
Tolerances:
  * fp32 outputs (LayerNorm z / out / d_res, stats, lse, loss): 1e-5 of the unit's largest reference magnitude -- fp32
    two-pass statistics over <= 2048 elements and the 2-ulp rsqrtf / __expf / __logf stay near 1e-6;
  * fp32 atomic reductions (dgamma, dbeta, d_words, d_positions, column sums): |err| <= 2e-5 * sum |terms| per column,
    which bounds the fp32 rounding of the terms and the summation order, whatever the order is;
  * bf16 outputs: max |err| <= 2^-7 * max |reference| of the unit (one bf16 rounding is 2^-9 relative);
  * masks, zero patterns, argmax indices, count_valid and untouched sentinels: exact.

The GPU tests run with `-m gpu`; the references themselves (against torch.autograd in fp64), the sensitivity of each
comparator to a one-element mistake, and argument rejection by the built library run without a device.
"""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

gpu = pytest.mark.gpu

BF16, F32, F64 = torch.bfloat16, torch.float32, torch.float64
# shapes of the configs: 30 caption positions, a 7 x 7 visual grid, a 10k vocabulary, 64-wide attention heads
T_CAP, SK, VOCAB, HEAD_DIM = 30, 49, 10000, 64
BF16_RTOL = 2.0 ** -7
F32_RTOL = 1e-5
SUM_RTOL = 2e-5


# ------------------------------------------------------------------------------------------------ dropout mask mirror
_MASK64 = (1 << 64) - 1
_GOLDEN = 0x9E3779B97F4A7C15
_MIX = np.uint64(0xD6E8FEB86659FD93)
_S32, _S16 = np.uint64(32), np.uint64(16)


def hash_u64(seed, site, ctr):
    """hash_u64 of csrc/vtx_common.cuh in numpy uint64 (array products wrap modulo 2^64 as in C)."""
    key = np.uint64((seed & _MASK64) ^ ((_GOLDEN * ((site + 1) & 0xFFFFFFFF)) & _MASK64))
    ctr = np.asarray(ctr, dtype=np.uint64)
    with np.errstate(over="ignore"):
        x = key ^ (ctr * _MIX)
        x = x ^ (x >> _S32)
        x = x * _MIX
        x = x ^ (x >> _S32)
        x = x * _MIX
        x = x ^ (x >> _S32)
    return x


def keep_scale(seed, site, flat_index, p):
    """Drop4 of csrc/vtx_common.cuh: 0 where element `flat_index` is dropped, float32 1 / (1 - p) where it is kept.
    One hash per flat_index >> 2; element flat_index & 3 of the group takes bits [16 * lane, 16 * lane + 16)."""
    idx = np.asarray(flat_index, dtype=np.uint64)
    if not p > 0:
        return np.ones(idx.shape, np.float32)
    p32 = np.float32(p)
    thr = np.uint32(p32 * np.float32(65536.0) + np.float32(0.5))
    inv_keep = np.float32(1.0) / (np.float32(1.0) - p32)
    h = hash_u64(seed, site, idx >> np.uint64(2))
    bits = (h >> (_S16 * (idx & np.uint64(3)))) & np.uint64(0xFFFF)
    return np.where(bits < np.uint64(thr), np.float32(0.0), inv_keep).astype(np.float32)


def keep_rows(seed, site, M, H, p, device="cpu"):
    """Mask of an elementwise [M, H] site (embedding, add + LN, ln_bwd, GELU): flat index row * H + col."""
    return torch.from_numpy(keep_scale(seed, site, np.arange(M * H, dtype=np.uint64), p)).view(M, H).to(device, F64)


def keep_attn(seed, site, B, heads, Tq, Tk, p, device="cpu"):
    """Mask of the attention probabilities: flat index ((b * heads + h) * 32 + i) * 64 + j."""
    u = np.arange(B * heads, dtype=np.uint64)[:, None, None]
    i = np.arange(Tq, dtype=np.uint64)[None, :, None]
    j = np.arange(Tk, dtype=np.uint64)[None, None, :]
    idx = (u * np.uint64(32) + i) * np.uint64(64) + j
    return torch.from_numpy(keep_scale(seed, site, idx, p)).view(B, heads, Tq, Tk).to(device, F64)


# ------------------------------------------------------------------------------------------------ fp64 references
def _bf(x):
    """Round to bf16 through fp32 (the kernels round fp32 values) and return in x's dtype."""
    return x.to(F32).to(BF16).to(x.dtype)


def ln_fwd_ref(z, gamma, beta, eps):
    mean = z.mean(1)
    var = ((z - mean[:, None]) ** 2).mean(1)
    rstd = 1.0 / torch.sqrt(var + eps)
    return (z - mean[:, None]) * rstd[:, None] * gamma + beta, mean, rstd


def ln_bwd_ref(g, z, mean, rstd, gamma):
    """LayerNorm backward from the saved statistics.  Returns dz, dgamma, dbeta and, for each, the sum of the absolute
    values of its terms (the scale its fp32 evaluation error is relative to)."""
    xh = (z - mean[:, None]) * rstd[:, None]
    dxh = g * gamma
    s1 = dxh.mean(1, keepdim=True)
    s2 = (dxh * xh).mean(1, keepdim=True)
    r = rstd[:, None]
    dz = r * (dxh - s1 - xh * s2)
    dz_mag = r.abs() * (dxh.abs() + s1.abs() + (xh * s2).abs())
    return dict(dz=dz, dz_mag=dz_mag, dgamma=(g * xh).sum(0), dgamma_mag=(g * xh).abs().sum(0), dbeta=g.sum(0),
                dbeta_mag=g.abs().sum(0))


def embed_fwd_ref(tokens, words, positions, gamma, beta, T, pad, eps, keep):
    t = torch.arange(tokens.numel(), device=tokens.device) % T
    z = words[tokens] + positions[t]
    out, mean, rstd = ln_fwd_ref(z, gamma, beta, eps)
    return z, mean, rstd, out * keep * (tokens != pad).to(out.dtype)[:, None]


def embed_bwd_ref(g, tokens, z, mean, rstd, gamma, T, pad, keep, V):
    """g = upstream gradient of the embedding output; scatter-adds of dz into the word and position tables."""
    t = torch.arange(tokens.numel(), device=tokens.device) % T
    g = g * keep * (tokens != pad).to(g.dtype)[:, None]
    r = ln_bwd_ref(g, z, mean, rstd, gamma)
    H = z.shape[1]
    zeros_w = torch.zeros(V, H, dtype=z.dtype, device=z.device)
    zeros_p = torch.zeros(T, H, dtype=z.dtype, device=z.device)
    r["d_words"] = zeros_w.clone().index_add_(0, tokens, r["dz"])
    r["d_words_mag"] = zeros_w.clone().index_add_(0, tokens, r["dz_mag"])
    r["d_pos"] = zeros_p.clone().index_add_(0, t, r["dz"])
    r["d_pos_mag"] = zeros_p.clone().index_add_(0, t, r["dz_mag"])
    return r


def attn_allowed(B, Tq, Tk, lengths, causal, device="cpu"):
    """[B, 1, Tq, Tk] key mask: causal 1 = j <= i and j < len, 2 = j < len, 0 = every key."""
    i = torch.arange(Tq, device=device)[None, :, None]
    j = torch.arange(Tk, device=device)[None, None, :]
    if causal == 0:
        ok = torch.ones(B, Tq, Tk, dtype=torch.bool, device=device)
    else:
        ok = j < lengths.to(device)[:, None, None]
        if causal == 1:
            ok = ok & (j <= i)
    return ok[:, None]


def attn_fwd_ref(q, k, v, allowed, keep, rounded=True):
    """q [B, h, Tq, 64], k / v [B, h, Tk, 64].  Returns out [B, h, Tq, 64] and lse [B, h, Tq]."""
    s = (q @ k.transpose(-1, -2)) * 0.125
    s = s.masked_fill(~allowed, -math.inf)
    mx = s.amax(-1, keepdim=True)
    e = torch.exp(s - mx)
    rsum = e.sum(-1, keepdim=True)
    pd = e * keep
    if rounded:
        pd = _bf(pd)
    out = (pd @ v) / rsum
    return out, (mx + torch.log(rsum)).squeeze(-1)


def attn_bwd_ref(q, k, v, do, allowed, keep, lse, rounded=True):
    s = (q @ k.transpose(-1, -2)) * 0.125
    p = torch.exp(s - lse[..., None]).masked_fill(~allowed, 0.0)
    dp = (do @ v.transpose(-1, -2)) * keep
    D = (p * dp).sum(-1, keepdim=True)
    ds = p * (dp - D) * 0.125
    pd = p * keep
    if rounded:
        ds, pd = _bf(ds), _bf(pd)
    return ds @ k, ds.transpose(-1, -2) @ q, pd.transpose(-1, -2) @ do


def gelu_ref(u):
    return 0.5 * u * (1.0 + torch.erf(u / math.sqrt(2.0)))


def gelu_grad_ref(u):
    return 0.5 * (1.0 + torch.erf(u / math.sqrt(2.0))) + u * torch.exp(-0.5 * u * u) / math.sqrt(2.0 * math.pi)


def ce_targets(tokens, pad, shift):
    """Target of every row (b, t): tokens[b, t + 1] (pad at t = T-1) when shift = 1, tokens[b, t] when shift = 0."""
    if shift:
        tgt = torch.cat([tokens[:, 1:], torch.full_like(tokens[:, :1], pad)], 1)
    else:
        tgt = tokens.clone()
    return tgt.reshape(-1)


def ce_ref(logits, tokens, pad, shift):
    """logits [B*T, V] fp64.  Returns sum of the per-row losses / n, dlogits (zero on ignored rows), the per-row
    losses and n = number of valid targets."""
    tgt = ce_targets(tokens, pad, shift)
    valid = tgt != pad
    n = int(valid.sum())
    lse = torch.logsumexp(logits, 1)
    rows = torch.arange(logits.shape[0], device=logits.device)
    nll = (lse - logits[rows, tgt.clamp(0, logits.shape[1] - 1)]) * valid
    inv_n = 1.0 / max(n, 1)
    grad = torch.softmax(logits, 1)
    grad[rows, tgt.clamp(0, logits.shape[1] - 1)] -= 1.0
    grad = grad * valid[:, None] * inv_n
    return nll.sum() * inv_n, grad, nll, n


def colsum_ref(x):
    return x.sum(0), x.abs().sum(0)


def argmax_ref(x):
    """First index of the row maximum, NaN counting as greater than every number (first NaN wins)."""
    nan = torch.isnan(x)
    first_nan = nan.to(torch.int32).argmax(1)
    mx = torch.where(nan, torch.full_like(x, -math.inf), x).amax(1, keepdim=True)
    first_max = (x == mx).to(torch.int32).argmax(1)
    return torch.where(nan.any(1), first_nan, first_max)


# ------------------------------------------------------------------------------------------------ per-unit comparators
def _worst(name, err, tol):
    """err, tol: [units]; prints and asserts the worst err / tol ratio."""
    ratio = torch.where(tol > 0, err / tol.clamp_min(1e-300), torch.where(err > 0, math.inf, 0.0))
    ratio = torch.nan_to_num(ratio, nan=math.inf)
    u = int(ratio.argmax())
    worst = float(ratio[u])
    print(f"{name}: worst err/tol = {worst:.3g} (unit {u} of {ratio.numel()})")
    assert worst <= 1.0, f"{name}: unit {u} err {float(err[u]):.3g} > tol {float(tol[u]):.3g}"


def check_units(name, out, ref, rtol, floor=0.0):
    """Units along dim 0: max |out - ref| <= rtol * max |ref| + floor within each unit."""
    out = out.detach().to(F64).reshape(out.shape[0], -1)
    ref = ref.detach().to(F64).reshape(ref.shape[0], -1).to(out.device)
    err = (out - ref).abs().amax(1)
    _worst(name, err, rtol * ref.abs().amax(1) + floor)


def check_bf16(name, out, ref):
    check_units(name, out, ref, BF16_RTOL)


def check_sum(name, out, ref, mag, rtol=SUM_RTOL):
    """Atomic reductions: every element is a unit; |out - ref| <= rtol * sum |terms|."""
    out = out.detach().to(F64).reshape(-1)
    err = (out - ref.to(out.device).reshape(-1)).abs()
    _worst(name, err, rtol * mag.to(out.device).reshape(-1))


def check_exact(name, out, ref):
    out, ref = out.detach().cpu(), ref.detach().cpu()
    bad = out != ref
    if out.is_floating_point():
        bad &= ~(torch.isnan(out.float()) & torch.isnan(ref.float()))
    print(f"{name}: {int(bad.sum())} of {bad.numel()} elements differ")
    assert not bad.any(), f"{name}: first mismatch at {bad.nonzero()[0].tolist()}"


def check_bits(name, out, ref):
    """Bit-identical tensors (NaN payloads, signed zeros and all)."""
    a = out.detach().cpu().contiguous()
    b = ref.detach().cpu().contiguous()
    it = {1: torch.uint8, 2: torch.int16, 4: torch.int32, 8: torch.int64}[a.element_size()]
    check_exact(name, a.view(it), b.view(it))


# ------------------------------------------------------------------------------------------------ GPU plumbing
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")


def _ops():
    from virtex_b200 import ops
    return ops


def _s():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return 0 if t is None else t.data_ptr()


def _seed(v):
    return torch.tensor([v], dtype=torch.int64, device="cuda")


# ------------------------------------------------------------------------------------------------ embedding
# (H, B, extra rows, p, upstream).  B * 30 is never a multiple of 4 for odd B; B = 256 (M = 7680) exceeds the
# 2 x SMs grid of the backward kernels, so rows wrap around the grid-stride loop; `extra` rows make M % T != 0 (the
# generic kernel at a register width).
EMB_CASES = [
    (128, 7, 0, 0.0, "a"), (256, 7, 0, 0.1, "b"), (512, 9, 0, 0.1, "ab"), (768, 7, 0, 0.0, "ab"),
    (1024, 5, 0, 0.1, "a"), (2048, 3, 0, 0.1, "b"), (1024, 7, 7, 0.1, "ab"), (512, 256, 0, 0.1, "ab"),
    (768, 256, 0, 0.1, "a"), (128, 256, 0, 0.0, "b"), (256, 256, 0, 0.1, "a"), (1024, 256, 0, 0.0, "ab"),
    (2048, 256, 0, 0.1, "ab"),
]


def _embed_inputs(H, M, T, V, pad, g):
    # 40 distinct tokens: repeats collide in the d_words scatter-add; the first 8 are "quiet" rows whose variance
    # (~2e-8) is comparable to eps = 1e-8, so a wrong epsilon changes their output
    pool = torch.randperm(V - 1, generator=g)[:40] + 1
    tokens = pool[torch.randint(0, 40, (M,), generator=g)]
    B = (M + T - 1) // T
    lens = torch.randint(1, T + 1, (B,), generator=g)
    lens[0] = T
    r = torch.arange(M)
    tokens[(r % T) >= lens[r // T]] = pad
    words = torch.randn(V, H, generator=g)
    words[pool[:8]] *= 1e-4
    positions = torch.randn(T, H, generator=g) * 1e-4
    gamma = torch.rand(H, generator=g) + 0.5
    beta = torch.randn(H, generator=g) * 0.3
    return tokens, words, positions, gamma, beta


@gpu
@pytest.mark.parametrize("H,B,extra,p,dy", EMB_CASES)
def test_embedding_forward_and_backward_match_fp64(H, B, extra, p, dy):
    _need_cuda()
    ops = _ops()
    T, V, pad, eps, site = T_CAP, VOCAB, 0, 1e-8, 3
    M = B * T + extra
    g = torch.Generator().manual_seed(H * 7919 + M)
    tokens, words, positions, gamma, beta = (x.cuda() for x in _embed_inputs(H, M, T, V, pad, g))
    seed = _seed(1234 + H)
    keep = keep_rows(1234 + H, site, M, H, p, "cuda")
    z = torch.full((M, H), math.nan, device="cuda")
    stats = torch.full((M, 2), math.nan, device="cuda")
    out = torch.full((M, H), math.nan, device="cuda")
    out_bf = torch.full((M, H), math.nan, dtype=BF16, device="cuda")
    ops.call("vtx_embed_fwd", tokens.data_ptr(), words.data_ptr(), positions.data_ptr(), gamma.data_ptr(),
             beta.data_ptr(), z.data_ptr(), stats.data_ptr(), out.data_ptr(), out_bf.data_ptr(), M, T, H, pad, eps, p,
             seed.data_ptr(), site, _s())
    zr, mean, rstd, outr = embed_fwd_ref(tokens, words.double(), positions.double(), gamma.double(), beta.double(), T,
                                         pad, eps, keep)
    check_units("embed z", z, zr, F32_RTOL)
    check_units("embed mean", stats[:, :1], mean[:, None], 0.0, F32_RTOL * zr.abs().amax(1))
    check_units("embed rstd", stats[:, 1:], rstd[:, None], F32_RTOL)
    check_units("embed out", out, outr, F32_RTOL)
    check_bits("embed out_bf == bf16(out)", out_bf, out.bfloat16())

    dy_a = torch.randn(M, H, generator=g).cuda() if "a" in dy else None
    dy_b = torch.randn(M, H, generator=g).bfloat16().cuda() if "b" in dy else None
    dw0 = (torch.randn(V, H, generator=g) * 0.1).cuda()
    dp0 = torch.randn(T, H, generator=g).cuda()
    dg0, db0 = torch.randn(H, generator=g).cuda(), torch.randn(H, generator=g).cuda()
    d_words, d_pos, d_gamma, d_beta = dw0.clone(), dp0.clone(), dg0.clone(), db0.clone()
    ops.call("vtx_embed_bwd", _p(dy_a), _p(dy_b), tokens.data_ptr(), z.data_ptr(), stats.data_ptr(), gamma.data_ptr(),
             d_words.data_ptr(), d_pos.data_ptr(), d_gamma.data_ptr(), d_beta.data_ptr(), M, T, H, pad, p,
             seed.data_ptr(), site, _s())
    up = torch.zeros(M, H, dtype=F64, device="cuda")
    if dy_a is not None:
        up += dy_a.double()
    if dy_b is not None:
        up += dy_b.double()
    r = embed_bwd_ref(up, tokens, z.double(), stats[:, 0].double(), stats[:, 1].double(), gamma.double(), T, pad,
                      keep, V)
    check_sum("embed d_words", d_words, dw0.double() + r["d_words"], dw0.double().abs() + r["d_words_mag"])
    check_sum("embed d_pos", d_pos, dp0.double() + r["d_pos"], dp0.double().abs() + r["d_pos_mag"])
    check_sum("embed d_gamma", d_gamma, dg0.double() + r["dgamma"], dg0.double().abs() + r["dgamma_mag"])
    check_sum("embed d_beta", d_beta, db0.double() + r["dbeta"], db0.double().abs() + r["dbeta_mag"])
    # rows of tokens that never occur, and the pad row, are not touched
    seen = torch.zeros(V, dtype=torch.bool, device="cuda")
    seen[tokens[tokens != pad]] = True
    check_bits("embed d_words untouched rows", d_words[~seen], dw0[~seen])


# ------------------------------------------------------------------------------------------------ add + LN, LN backward
# (H, M, ln, inputs, outputs, p, upstream, skip): inputs r = residual, b = bf16 branch; outputs both / out / bf;
# skip none / sep (a separate d_skip) / alias (d_skip == d_res, as the pre-norm backward passes them) / nores
# (d_res NULL).  M = 7680 exceeds the 2 x SMs grid of the backward kernels.
LN_CASES = [
    (128, 210, 1, "rb", "both", 0.1, "ab", "none"), (256, 150, 1, "r", "out", 0.0, "b", "sep"),
    (512, 270, 1, "b", "bf", 0.1, "a", "alias"), (768, 210, 1, "rb", "both", 0.1, "ab", "nores"),
    (1024, 90, 1, "rb", "bf", 0.1, "b", "alias"), (2048, 150, 1, "rb", "both", 0.0, "ab", "sep"),
    (512, 7680, 1, "rb", "both", 0.1, "ab", "none"), (768, 7680, 1, "rb", "out", 0.1, "b", "alias"),
    (2048, 7680, 1, "r", "bf", 0.0, "a", "none"), (1024, 7680, 1, "b", "both", 0.1, "a", "sep"),
    (128, 90, 1, "r", "both", 0.0, "ab", "nores"), (256, 7680, 1, "rb", "both", 0.1, "ab", "alias"),
    (128, 7680, 0, "rb", "out", 0.1, "a", "none"), (256, 210, 0, "b", "both", 0.1, "ab", "sep"),
    (768, 150, 0, "rb", "bf", 0.1, "a", "alias"), (2048, 90, 0, "r", "both", 0.0, "b", "none"),
]


@gpu
@pytest.mark.parametrize("H,M,ln,src,outs,p,dy,skip", LN_CASES)
def test_add_layernorm_forward_and_backward_match_fp64(H, M, ln, src, outs, p, dy, skip):
    _need_cuda()
    ops = _ops()
    eps, site = 1e-5, 21
    g = torch.Generator().manual_seed(H * 31 + M + 7 * ln)
    # every 5th row is "quiet": variance ~1e-5, comparable to eps
    scale = torch.where(torch.arange(M) % 5 == 0, 3e-3, 1.0)[:, None]
    res = (torch.randn(M, H, generator=g) * scale).cuda() if "r" in src else None
    branch = (torch.randn(M, H, generator=g) * scale).bfloat16().cuda() if "b" in src else None
    gamma = (torch.rand(H, generator=g) + 0.5).cuda()
    beta = (torch.randn(H, generator=g) * 0.3).cuda()
    seed = _seed(99 + H)
    keep = keep_rows(99 + H, site, M, H, p, "cuda")
    z = torch.full((M, H), math.nan, device="cuda")
    stats = torch.full((M, 2), math.nan, device="cuda")
    out = torch.full((M, H), math.nan, device="cuda") if outs in ("both", "out") else None
    out_bf = torch.full((M, H), math.nan, dtype=BF16, device="cuda") if outs in ("both", "bf") else None
    ops.call("vtx_add_ln_fwd", _p(res), _p(branch), gamma.data_ptr() if ln else 0, beta.data_ptr() if ln else 0,
             z.data_ptr(), stats.data_ptr() if ln else 0, _p(out), _p(out_bf), M, H, eps, p, seed.data_ptr(), site, ln,
             _s())
    zr = torch.zeros(M, H, dtype=F64, device="cuda")
    if res is not None:
        zr += res.double()
    if branch is not None:
        zr += branch.double() * keep
    check_units("add_ln z", z, zr, F32_RTOL)
    if ln:
        outr, mean, rstd = ln_fwd_ref(zr, gamma.double(), beta.double(), eps)
        check_units("add_ln mean", stats[:, :1], mean[:, None], 0.0, F32_RTOL * zr.abs().amax(1))
        check_units("add_ln rstd", stats[:, 1:], rstd[:, None], F32_RTOL)
    else:
        outr = zr
    if out is not None:
        check_units("add_ln out", out, outr, F32_RTOL)
    if out_bf is not None:
        if out is not None:
            check_bits("add_ln out_bf == bf16(out)", out_bf, out.bfloat16())
        else:
            check_bf16("add_ln out_bf", out_bf, outr)

    # backward: g = dy_a + dy_b -> (LN backward) -> dz;  d_res = dz + d_skip;  d_branch = bf16(dz * mask)
    dy_a = torch.randn(M, H, generator=g).cuda() if "a" in dy else None
    dy_b = torch.randn(M, H, generator=g).bfloat16().cuda() if "b" in dy else None
    skip0 = torch.randn(M, H, generator=g).cuda()
    d_res = {"nores": None, "alias": skip0.clone()}.get(skip, torch.full((M, H), math.nan, device="cuda"))
    d_skip = {"sep": skip0, "alias": d_res}.get(skip)
    d_branch = torch.full((M, H), math.nan, dtype=BF16, device="cuda")
    dg0, db0 = torch.randn(H, generator=g).cuda(), torch.randn(H, generator=g).cuda()
    d_gamma, d_beta = dg0.clone(), db0.clone()
    ops.call("vtx_ln_bwd", _p(dy_a), _p(dy_b), z.data_ptr() if ln else 0, stats.data_ptr() if ln else 0,
             gamma.data_ptr() if ln else 0, _p(d_skip), _p(d_res), d_branch.data_ptr(), d_gamma.data_ptr() if ln else 0,
             d_beta.data_ptr() if ln else 0, M, H, p, seed.data_ptr(), site, ln, _s())
    up = torch.zeros(M, H, dtype=F64, device="cuda")
    if dy_a is not None:
        up += dy_a.double()
    if dy_b is not None:
        up += dy_b.double()
    if ln:
        r = ln_bwd_ref(up, z.double(), stats[:, 0].double(), stats[:, 1].double(), gamma.double())
        dz = r["dz"]
        check_sum("ln_bwd d_gamma", d_gamma, dg0.double() + r["dgamma"], dg0.double().abs() + r["dgamma_mag"])
        check_sum("ln_bwd d_beta", d_beta, db0.double() + r["dbeta"], db0.double().abs() + r["dbeta_mag"])
    else:
        dz = up
        check_bits("ln_bwd d_gamma untouched (ln = 0)", d_gamma, dg0)
        check_bits("ln_bwd d_beta untouched (ln = 0)", d_beta, db0)
    if d_res is not None:
        check_units("ln_bwd d_res", d_res, dz + (skip0.double() if d_skip is not None else 0.0), F32_RTOL)
    check_bf16("ln_bwd d_branch", d_branch, dz * keep)
    check_exact("ln_bwd d_branch zero where dropped", d_branch.float()[keep == 0] != 0,
                torch.zeros(int((keep == 0).sum()), dtype=torch.bool))
    if d_res is not None and d_skip is None:
        # the dropped / scaled branch gradient is the kernel's own fp32 dz times the mask, rounded once
        check_bits("ln_bwd d_branch == bf16(dz * keep)", d_branch, (d_res * keep.float()).bfloat16())


# ------------------------------------------------------------------------------------------------ attention
ATTN_SHAPES = [(T_CAP, T_CAP), (T_CAP, SK), (13, 13), (2, 2), (32, 64), (1, 17)]
ATTN_HEADS = [2, 8, 12, 16, 32]
# batch per head count: B * heads is not a multiple of 3 (warps per backward block) except for 12 heads, and not a
# multiple of 4 (warps per forward block) for 2 heads; 8, 16 and 32 heads are always multiples of 4
ATTN_BATCH = {2: 7, 8: 5, 12: 3, 16: 5, 32: 2}
ATTN_CASES = [(c, tq, tk, ATTN_HEADS[(3 * k + c) % 5], p)
              for k, (tq, tk) in enumerate(ATTN_SHAPES) for c in (0, 1, 2) for p in (0.0, 0.1)]
_SENT = -777.0  # bf16-exact sentinel of the output buffers


def _attn_lengths(B, Tq, Tk, c):
    cand = [1, 2, Tq, max(1, Tq // 2), Tk, max(1, Tq - 1), 3]
    return torch.tensor([min(max(cand[(b + c) % len(cand)], 1), Tk) for b in range(B)], dtype=torch.int64)


def _heads_view(x, B, T, heads, col0):
    """[B*T, ld] packed rows -> [B, heads, T, 64] of the columns [col0, col0 + heads * 64)."""
    return x[:, col0:col0 + heads * HEAD_DIM].reshape(B, T, heads, HEAD_DIM).permute(0, 2, 1, 3)


@gpu
@pytest.mark.parametrize("causal,Tq,Tk,heads,p", ATTN_CASES)
def test_attention_forward_and_backward_match_fp64(causal, Tq, Tk, heads, p):
    _need_cuda()
    ops = _ops()
    B = ATTN_BATCH[heads]
    H = heads * HEAD_DIM
    site = 7
    g = torch.Generator().manual_seed(1000 * causal + 37 * Tq + Tk + heads)
    lengths = _attn_lengths(B, Tq, Tk, causal).cuda()
    e = 2  # bytes per bf16
    if Tq == Tk:  # self-attention layout: packed qkv [B*T, 3H]
        qkv = (torch.randn(B * Tq, 3 * H, generator=g) * 0.7).bfloat16().cuda()
        qp, kp, vp, ldq, ldk = qkv.data_ptr(), qkv.data_ptr() + H * e, qkv.data_ptr() + 2 * H * e, 3 * H, 3 * H
        q, k, v = (_heads_view(qkv, B, Tq, heads, c0) for c0 in (0, H, 2 * H))
    else:  # cross-attention layout: q [B*Tq, H], packed kv [B*Tk, 2H]
        qc = (torch.randn(B * Tq, H, generator=g) * 0.7).bfloat16().cuda()
        kv = (torch.randn(B * Tk, 2 * H, generator=g) * 0.7).bfloat16().cuda()
        qp, kp, vp, ldq, ldk = qc.data_ptr(), kv.data_ptr(), kv.data_ptr() + H * e, H, 2 * H
        q = _heads_view(qc, B, Tq, heads, 0)
        k, v = (_heads_view(kv, B, Tk, heads, c0) for c0 in (0, H))
    gap = 0 if p == 0 else 16  # extra columns of the output buffers: they, and two extra rows, must stay sentinel
    ldo = H + gap
    obuf = torch.full((B * Tq + 2, ldo), _SENT, dtype=BF16, device="cuda")
    lse = torch.full((B * heads * 32,), 1234.5, device="cuda")
    seed = _seed(4242 + heads)
    keep = keep_attn(4242 + heads, site, B, heads, Tq, Tk, p, "cuda")
    allowed = attn_allowed(B, Tq, Tk, lengths, causal, "cuda")
    lens_ptr = lengths.data_ptr() if causal else 0
    ops.call("vtx_attn_fwd", qp, ldq, kp, ldk, vp, ldk, obuf.data_ptr(), ldo, lse.data_ptr(), B, heads, Tq, Tk,
             lens_ptr, causal, p, seed.data_ptr(), site, _s())
    q64, k64, v64 = q.double(), k.double(), v.double()
    o_ref, lse_ref = attn_fwd_ref(q64, k64, v64, allowed, keep)
    units = B * heads
    check_bf16("attn out", _heads_view(obuf[:B * Tq], B, Tq, heads, 0).reshape(units, -1), o_ref.reshape(units, -1))
    lse_k = lse.view(B, heads, 32)
    # lse is a logarithm: its fp32 error is absolute, hence the floor of 1e-5
    check_units("attn lse", lse_k[..., :Tq].reshape(units, -1), lse_ref.reshape(units, -1), F32_RTOL, F32_RTOL)
    check_bits("attn lse rows >= Tq untouched", lse_k[..., Tq:], torch.full_like(lse_k[..., Tq:], 1234.5))
    outside = obuf.clone()
    outside[:B * Tq, :H] = _SENT
    check_bits("attn out outside the heads' columns untouched", outside, torch.full_like(obuf, _SENT))

    do = (torch.randn(B * Tq, H, generator=g)).bfloat16().cuda()
    if Tq == Tk:
        ldd = 3 * H + gap
        dbuf = torch.full((B * Tq + 2, ldd), _SENT, dtype=BF16, device="cuda")
        dqp, dkp, dvp, lddq, lddk = dbuf.data_ptr(), dbuf.data_ptr() + H * e, dbuf.data_ptr() + 2 * H * e, ldd, ldd
        bufs = [(dbuf, B * Tq, 3 * H)]
        dq_v, dk_v, dv_v = (_heads_view(dbuf[:B * Tq], B, Tq, heads, c0) for c0 in (0, H, 2 * H))
    else:
        dqb = torch.full((B * Tq + 2, H + gap), _SENT, dtype=BF16, device="cuda")
        dkvb = torch.full((B * Tk + 2, 2 * H + gap), _SENT, dtype=BF16, device="cuda")
        dqp, dkp, dvp, lddq, lddk = dqb.data_ptr(), dkvb.data_ptr(), dkvb.data_ptr() + H * e, H + gap, 2 * H + gap
        bufs = [(dqb, B * Tq, H), (dkvb, B * Tk, 2 * H)]
        dq_v = _heads_view(dqb[:B * Tq], B, Tq, heads, 0)
        dk_v, dv_v = (_heads_view(dkvb[:B * Tk], B, Tk, heads, c0) for c0 in (0, H))
    ops.call("vtx_attn_bwd", qp, ldq, kp, ldk, vp, ldk, do.data_ptr(), H, lse.data_ptr(), dqp, lddq, dkp, lddk, dvp,
             lddk, B, heads, Tq, Tk, lens_ptr, causal, p, seed.data_ptr(), site, _s())
    dq_r, dk_r, dv_r = attn_bwd_ref(q64, k64, v64, _heads_view(do, B, Tq, heads, 0).double(), allowed, keep, lse_ref)
    check_bf16("attn dq", dq_v.reshape(units, -1), dq_r.reshape(units, -1))
    check_bf16("attn dk", dk_v.reshape(units, -1), dk_r.reshape(units, -1))
    check_bf16("attn dv", dv_v.reshape(units, -1), dv_r.reshape(units, -1))
    for buf, rows, cols in bufs:
        outside = buf.clone()
        outside[:rows, :cols] = _SENT
        check_bits("attn grads outside the blocks untouched", outside, torch.full_like(buf, _SENT))


# ------------------------------------------------------------------------------------------------ GELU + dropout
# n = M * 4H at the configs' sizes; every case but the second exceeds the 8 x SMs x 256 x 8-element grid, so the
# grid-stride loop runs several rounds
GELU_CASES = [(1920, 4096, 0.1), (210, 512, 0.0), (7680, 3072, 0.1), (150, 8192, 0.1)]


def check_ulps(name, out, ref, sel, max_frac):
    """bf16 `out` within one ulp of `ref` on the elements `sel`, and at most `max_frac` of them not bit-identical."""
    a = out.view(torch.int16)[sel].to(torch.int32)
    b = ref.to(F32).to(BF16).view(torch.int16)[sel].to(torch.int32)
    d = (a - b).abs()
    frac = float((d > 0).double().mean()) if d.numel() else 0.0
    worst = int(d.max()) if d.numel() else 0
    print(f"{name}: {frac:.2e} of {d.numel()} elements one ulp off (limit {max_frac:g}), max {worst} ulp")
    assert worst <= 1, name
    assert frac <= max_frac, name


@gpu
@pytest.mark.parametrize("M,Fd,p", GELU_CASES)
def test_gelu_dropout_forward_and_in_place_backward_match_fp64(M, Fd, p):
    _need_cuda()
    ops = _ops()
    n, site = M * Fd, 14
    gen = torch.Generator(device="cuda").manual_seed(M + Fd)
    u = (torch.randn(M, Fd, generator=gen, device="cuda") * 1.5).bfloat16()
    h = torch.full((M, Fd), math.nan, dtype=BF16, device="cuda")
    seed = _seed(77)
    keep = keep_rows(77, site, M, Fd, p, "cuda")
    ops.call("vtx_gelu_dropout_fwd", u.data_ptr(), h.data_ptr(), n, p, seed.data_ptr(), site, _s())
    u64 = u.double()
    h_ref = _bf(_bf(gelu_ref(u64)) * keep)
    check_bf16("gelu fwd", h, h_ref)
    # the mirror reproduces the kernel's mask exactly: zeros where dropped, non-zero where kept (|u| < 3, where the
    # fp32 gelu cannot underflow)
    kept_live = (keep != 0) & (u64 != 0) & (u64.abs() < 3)
    check_exact("gelu fwd dropped elements are zero", h[keep == 0].float(), torch.zeros(int((keep == 0).sum())))
    check_exact("gelu fwd kept elements are non-zero", h[kept_live] != 0,
                torch.ones(int(kept_live.sum()), dtype=torch.bool))
    # |u| < 3: 1 + erff(u / sqrt 2) keeps >= 16 significant bits in fp32, so the kernel's erff can only flip the bf16
    # rounding of gelu(u) to a neighbour, and rarely
    check_ulps("gelu fwd ulps", h, h_ref, kept_live, 1e-3)

    dh = torch.randn(M, Fd, generator=gen, device="cuda").bfloat16()
    dh0 = dh.clone()
    ops.call("vtx_gelu_dropout_bwd", dh.data_ptr(), u.data_ptr(), dh.data_ptr(), n, p, seed.data_ptr(), site, _s())
    gp = gelu_grad_ref(u64)
    du_ref = _bf(dh0.double() * keep * gp)
    check_bf16("gelu bwd (in place)", dh, du_ref)
    check_exact("gelu bwd dropped elements are zero", dh[keep == 0].float(), torch.zeros(int((keep == 0).sum())))
    # away from the root of gelu' (u ~ -0.75), where Phi(u) + u phi(u) cancels
    check_ulps("gelu bwd ulps", dh, du_ref, (keep != 0) & (u64.abs() < 3) & (gp.abs() > 1e-2) & (dh0 != 0), 1e-3)


# ------------------------------------------------------------------------------------------------ cross entropy
# (V, ldl, B, shift, pad): V = 10240 is the largest row of the register kernel ce_reg_kernel<5>, 10248 and 16384 run
# the generic ce_kernel; B * 30 = 8400 > 8192 makes count_valid's 32 x 256-thread grid-stride loop wrap
CE_CASES = [(8, 16, 3, 1, 2), (1000, 1000, 5, 1, 0), (10000, 10000, 280, 1, 0), (10240, 10248, 5, 0, 2),
            (10248, 10256, 5, 1, 2), (16384, 16384, 3, 0, 0)]


@gpu
@pytest.mark.parametrize("V,ldl,B,shift,pad", CE_CASES)
def test_cross_entropy_and_count_valid_match_fp64(V, ldl, B, shift, pad):
    _need_cuda()
    ops = _ops()
    T = T_CAP
    R = B * T
    g = torch.Generator().manual_seed(V + B + shift)
    tokens = torch.randint(0, V, (B, T), generator=g)
    lens = torch.randint(2, T + 1, (B,), generator=g)
    lens[0] = T
    tokens[torch.arange(T)[None] >= lens[:, None]] = pad
    tokens[1] = pad                      # a caption of nothing but padding
    tokens[0, 1], tokens[0, 2] = 0, V - 1  # targets at both ends of the vocabulary
    tokens = tokens.cuda()
    gen = torch.Generator(device="cuda").manual_seed(V)
    lg = torch.randn(R, ldl, generator=gen, device="cuda") * 3
    lg[::7] *= 20                        # logits of magnitude ~60
    lg[:, V:] = 3e4                      # past the row end: a read there would dominate the softmax
    logits = lg.bfloat16()
    logits0 = logits.clone()
    count = torch.zeros(1, device="cuda")
    loss = torch.full((1,), 1.25, device="cuda")
    L_ref, grad_ref, nll, n = ce_ref(logits0[:, :V].double(), tokens, pad, shift)
    ops.call("vtx_count_valid", tokens.data_ptr(), B, T, pad, shift, count.data_ptr(), _s())
    check_exact("count_valid", count.cpu(), torch.tensor([float(n)]))
    ops.call("vtx_cross_entropy", logits.data_ptr(), ldl, tokens.data_ptr(), B, T, V, pad, shift, count.data_ptr(),
             loss.data_ptr(), 0, _s())
    check_bits("cross_entropy write_grad = 0 leaves the logits", logits, logits0)
    # the loss is one fp32 atomic sum of per-row terms; tolerance relative to the sum of their magnitudes
    mag = nll.abs().sum() / max(n, 1)
    _worst("cross_entropy loss", (loss.double() - (1.25 + L_ref)).abs().cpu(), (F32_RTOL * (1.25 + mag)).view(1).cpu())
    ops.call("vtx_cross_entropy", logits.data_ptr(), ldl, tokens.data_ptr(), B, T, V, pad, shift, count.data_ptr(),
             loss.data_ptr(), 1, _s())
    _worst("cross_entropy loss accumulates", (loss.double() - (1.25 + 2 * L_ref)).abs().cpu(),
           (F32_RTOL * (1.25 + 2 * mag)).view(1).cpu())
    # per row; rows without a target must be exactly zero (their tolerance is 0)
    check_bf16("cross_entropy dlogits", logits[:, :V], grad_ref)
    check_bits("cross_entropy columns past V untouched", logits[:, V:], logits0[:, V:])
    ops.call("vtx_count_valid", tokens.data_ptr(), B, T, pad, shift, count.data_ptr(), _s())
    check_exact("count_valid accumulates", count.cpu(), torch.tensor([2.0 * n]))


@gpu
@pytest.mark.parametrize("shift", [0, 1])
def test_cross_entropy_without_valid_targets_keeps_the_loss_and_zeroes_the_gradient(shift):
    _need_cuda()
    ops = _ops()
    V, B, T, pad = 1000, 3, T_CAP, 0
    tokens = torch.full((B, T), pad, dtype=torch.int64, device="cuda")
    if shift:
        tokens[:, 0] = 5  # position 0 is never a next-token target
    logits = torch.randn(B * T, V, device="cuda").bfloat16()
    count = torch.zeros(1, device="cuda")
    loss = torch.full((1,), 0.5, device="cuda")
    ops.call("vtx_count_valid", tokens.data_ptr(), B, T, pad, shift, count.data_ptr(), _s())
    ops.call("vtx_cross_entropy", logits.data_ptr(), V, tokens.data_ptr(), B, T, V, pad, shift, count.data_ptr(),
             loss.data_ptr(), 1, _s())
    check_bits("count_valid of an all-pad batch", count, torch.zeros(1))
    check_bits("loss unchanged", loss, torch.full((1,), 0.5))
    check_bits("dlogits all zero", logits, torch.zeros_like(logits))


# ------------------------------------------------------------------------------------------------ column sums
# M on both sides of the M >= 64 threshold of colsum_lanes_kernel; N = 100 (ld 104) is not a multiple of 8 and runs
# colsum_kernel at every M.  M = 30 B / 49 B are the head's bias-gradient rows at batch 1.
COLSUM_M = [1, 30, 49, 63, 64, 65, 7680, 12544]
COLSUM_N = [(64, 64), (200, 224), (1000, 1000), (2048, 2072), (3072, 3072), (10000, 10000), (100, 104)]


@gpu
@pytest.mark.parametrize("N,ld", COLSUM_N)
@pytest.mark.parametrize("M", COLSUM_M)
def test_colsum_matches_fp64(M, N, ld):
    _need_cuda()
    ops = _ops()
    gen = torch.Generator(device="cuda").manual_seed(7 * M + N)
    x = torch.randn(M, ld, generator=gen, device="cuda").bfloat16()
    x[:, N:] = 1e4  # past the row end: must not be summed
    out0 = torch.randn(N, generator=gen, device="cuda")
    out = out0.clone()
    ops.call("vtx_colsum", x.data_ptr(), ld, M, N, out.data_ptr(), _s())
    s, mag = colsum_ref(x[:, :N].double())
    check_sum(f"colsum M={M} N={N}", out, out0.double() + s, out0.double().abs() + mag)


# ------------------------------------------------------------------------------------------------ argmax
def _argmax_input(N, ld, g):
    x = torch.randn(12, ld, generator=g)
    x[:, N:] = math.nan                  # past the row end: a read there would win
    big = float(x[:, :N].abs().max()) + 1
    x[1, N // 3] = x[1, N - 1] = big     # a tie: the first index wins
    x[2, :N] = -math.inf                 # all -inf: index 0
    x[3, 0] = 1e30                       # some NaNs after the largest finite value: the first NaN wins
    x[3, N // 2] = x[3, N - 1] = math.nan
    x[4, :N] = math.nan                  # all NaN: index 0
    x[5, :N] = 2.5                       # constant row: index 0
    x[6, N - 1] = math.nan               # NaN in the last column only
    x[7, 0], x[7, N - 1] = math.inf, math.nan
    x[8, :N] = -math.inf
    x[8, N // 2] = math.nan
    x[9, N // 4] = x[9, N - 1] = math.inf
    return x


@gpu
@pytest.mark.parametrize("N,ld", [(1, 8), (255, 264), (256, 256), (10000, 10008)])
def test_argmax_rows_matches_torch_argmax(N, ld):
    _need_cuda()
    ops = _ops()
    x = _argmax_input(N, ld, torch.Generator().manual_seed(N))
    xd = x.cuda()
    out = torch.full((x.shape[0],), -5, dtype=torch.int64, device="cuda")
    ops.call("vtx_argmax_rows", xd.data_ptr(), ld, x.shape[0], N, out.data_ptr(), _s())
    check_exact(f"argmax N={N} vs torch.argmax", out.cpu(), torch.argmax(x[:, :N], 1))
    check_exact(f"argmax N={N} vs reference", out.cpu(), argmax_ref(x[:, :N]))


# ------------------------------------------------------------------------------------------------ CPU: the references
def test_keep_scale_rate_scale_and_grouping():
    idx = np.arange(1 << 16, dtype=np.uint64)
    k = keep_scale(5, 3, idx, 0.1)
    assert set(np.unique(k).tolist()) == {0.0, float(np.float32(1) / (np.float32(1) - np.float32(0.1)))}
    rate = float((k == 0).mean())
    assert abs(rate - 6554 / 65536) < 3 * math.sqrt(0.1 * 0.9 / idx.size)
    assert np.array_equal(keep_scale(5, 3, idx, 0.1), k) and not np.array_equal(keep_scale(6, 3, idx, 0.1), k)
    assert (keep_scale(5, 3, idx, 0.0) == 1).all()
    # four consecutive elements share one hash: element 4q + l depends only on (q, l)
    assert np.array_equal(keep_scale(5, 3, idx[4:8], 0.1), k[4:8])
    h = hash_u64(5, 3, np.uint64(1))
    assert k[5] == (0.0 if ((int(h) >> 16) & 0xFFFF) < 6554 else k.max())


def test_layernorm_reference_matches_autograd():
    g = torch.Generator().manual_seed(0)
    z = torch.randn(6, 256, dtype=F64, generator=g)
    z[0] *= 1e-4
    gamma = torch.rand(256, dtype=F64, generator=g) + 0.5
    beta = torch.randn(256, dtype=F64, generator=g)
    dy = torch.randn(6, 256, dtype=F64, generator=g)
    for eps in (1e-8, 1e-5):
        zr, gr, br = (t.clone().requires_grad_(True) for t in (z, gamma, beta))
        y = F.layer_norm(zr, (256,), gr, br, eps)
        y.backward(dy)
        out, mean, rstd = ln_fwd_ref(z, gamma, beta, eps)
        torch.testing.assert_close(out, y.detach(), rtol=1e-10, atol=1e-12)
        r = ln_bwd_ref(dy, z, mean, rstd, gamma)
        torch.testing.assert_close(r["dz"], zr.grad, rtol=1e-9, atol=1e-9)
        torch.testing.assert_close(r["dgamma"], gr.grad, rtol=1e-10, atol=1e-10)
        torch.testing.assert_close(r["dbeta"], br.grad, rtol=1e-10, atol=1e-10)


def test_embedding_reference_matches_autograd():
    g = torch.Generator().manual_seed(1)
    V, T, H, pad, p = 50, 6, 128, 0, 0.1
    tokens = torch.randint(0, 8, (4 * T,), generator=g)  # repeats, and pad = 0
    words = torch.randn(V, H, dtype=F64, generator=g)
    positions = torch.randn(T, H, dtype=F64, generator=g)
    gamma = torch.rand(H, dtype=F64, generator=g) + 0.5
    beta = torch.randn(H, dtype=F64, generator=g)
    keep = keep_rows(9, 2, tokens.numel(), H, p)
    dy = torch.randn(tokens.numel(), H, dtype=F64, generator=g)
    w, ps, gm, bt = (t.clone().requires_grad_(True) for t in (words, positions, gamma, beta))
    t = torch.arange(tokens.numel()) % T
    y = F.layer_norm(w[tokens] + ps[t], (H,), gm, bt, 1e-8) * keep * (tokens != pad).double()[:, None]
    y.backward(dy)
    z, mean, rstd, out = embed_fwd_ref(tokens, words, positions, gamma, beta, T, pad, 1e-8, keep)
    torch.testing.assert_close(out, y.detach(), rtol=1e-10, atol=1e-12)
    r = embed_bwd_ref(dy, tokens, z, mean, rstd, gamma, T, pad, keep, V)
    for name, ref in (("d_words", w.grad), ("d_pos", ps.grad), ("dgamma", gm.grad), ("dbeta", bt.grad)):
        torch.testing.assert_close(r[name], ref, rtol=1e-9, atol=1e-9, msg=name)


@pytest.mark.parametrize("causal,Tq,Tk", [(0, 5, 7), (1, 6, 6), (2, 6, 6), (1, 3, 9)])
def test_attention_reference_matches_autograd(causal, Tq, Tk):
    g = torch.Generator().manual_seed(causal)
    B, heads = 3, 2
    lengths = torch.tensor([1, 3, Tk])
    q, k, v, do = (torch.randn(B, heads, n, HEAD_DIM, dtype=F64, generator=g) for n in (Tq, Tk, Tk, Tq))
    keep = keep_attn(3, 4, B, heads, Tq, Tk, 0.1)
    allowed = attn_allowed(B, Tq, Tk, lengths, causal)
    qr, kr, vr = (t.clone().requires_grad_(True) for t in (q, k, v))
    s = (qr @ kr.transpose(-1, -2) * 0.125).masked_fill(~allowed, -math.inf)
    o = (torch.softmax(s, -1) * keep) @ vr
    o.backward(do)
    o_ref, lse = attn_fwd_ref(q, k, v, allowed, keep, rounded=False)
    torch.testing.assert_close(o_ref, o.detach(), rtol=1e-10, atol=1e-12)
    torch.testing.assert_close(lse, torch.logsumexp(s.detach(), -1), rtol=1e-12, atol=1e-12)
    dq, dk, dv = attn_bwd_ref(q, k, v, do, allowed, keep, lse, rounded=False)
    for name, a, b in (("dq", dq, qr.grad), ("dk", dk, kr.grad), ("dv", dv, vr.grad)):
        torch.testing.assert_close(a, b, rtol=1e-9, atol=1e-10, msg=name)


def test_gelu_reference_matches_autograd():
    u = torch.linspace(-8, 8, 4001, dtype=F64).requires_grad_(True)
    y = F.gelu(u)
    y.sum().backward()
    torch.testing.assert_close(gelu_ref(u.detach()), y.detach(), rtol=1e-12, atol=1e-15)
    torch.testing.assert_close(gelu_grad_ref(u.detach()), u.grad, rtol=1e-12, atol=1e-15)


@pytest.mark.parametrize("shift,pad", [(1, 0), (0, 2)])
def test_cross_entropy_reference_matches_torch(shift, pad):
    g = torch.Generator().manual_seed(shift)
    B, T, V = 3, 7, 40
    tokens = torch.randint(0, V, (B, T), generator=g)
    tokens[1] = pad
    tokens[2, 4:] = pad
    logits = (torch.randn(B * T, V, dtype=F64, generator=g) * 5).requires_grad_(True)
    tgt = ce_targets(tokens, pad, shift)
    n = int((tgt != pad).sum())
    L = F.cross_entropy(logits, tgt, ignore_index=pad, reduction="sum") / n
    L.backward()
    L_ref, grad, _, n_ref = ce_ref(logits.detach(), tokens, pad, shift)
    assert n_ref == n
    torch.testing.assert_close(L_ref, L.detach(), rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(grad, logits.grad, rtol=1e-10, atol=1e-12)


def test_argmax_reference_matches_torch_argmax():
    for N, ld in ((1, 8), (255, 264), (256, 256)):
        x = _argmax_input(N, ld, torch.Generator().manual_seed(N))[:, :N]
        assert torch.equal(argmax_ref(x), torch.argmax(x, 1))


# ------------------------------------------------------------------------------------------------ CPU: sensitivity
# Each comparator accepts an fp32 evaluation of the same formula (what a correct kernel produces) and rejects the
# reference with one deliberate mistake.
def _attn_case():
    g = torch.Generator().manual_seed(11)
    B, heads, T = 2, 2, 8
    q, k, v, do = (_bf(torch.randn(B, heads, T, HEAD_DIM, dtype=F64, generator=g) * 0.7) for _ in range(4))
    lengths = torch.tensor([8, 6])
    return q, k, v, do, attn_allowed(B, T, T, lengths, 1), keep_attn(1, 2, B, heads, T, T, 0.1)


@pytest.mark.parametrize("mistake", ["extra key", "missing key"])
def test_attention_comparator_rejects_one_wrong_key(mistake):
    q, k, v, do, allowed, keep = _attn_case()
    units = q.shape[0] * q.shape[1]
    o_ref, lse = attn_fwd_ref(q, k, v, allowed, keep)
    dq_ref = attn_bwd_ref(q, k, v, do, allowed, keep, lse)[0]
    o32, lse32 = attn_fwd_ref(q.float(), k.float(), v.float(), allowed, keep.float())
    dq32 = attn_bwd_ref(q.float(), k.float(), v.float(), do.float(), allowed, keep.float(), lse32)[0]
    check_bf16("fp32 attention out", _bf(o32).reshape(units, -1), o_ref.reshape(units, -1))
    check_bf16("fp32 attention dq", _bf(dq32).reshape(units, -1), dq_ref.reshape(units, -1))
    bad = allowed.expand(-1, q.shape[1], -1, -1).clone()
    if mistake == "extra key":
        bad[0, 1, 2, 3] = True   # row 2 of a causal block sees key 3
    else:
        bad[1, 0, 4, 0] = False  # row 4 loses key 0
    o_bad, lse_bad = attn_fwd_ref(q, k, v, bad, keep)
    with pytest.raises(AssertionError):
        check_bf16("attention out, one wrong key", _bf(o_bad).reshape(units, -1), o_ref.reshape(units, -1))
    dq_bad = attn_bwd_ref(q, k, v, do, bad, keep, lse_bad)[0]
    with pytest.raises(AssertionError):
        check_bf16("attention dq, one wrong key", _bf(dq_bad).reshape(units, -1), dq_ref.reshape(units, -1))


def test_layernorm_comparator_rejects_the_wrong_epsilon():
    g = torch.Generator().manual_seed(2)
    z = torch.randn(8, 512, generator=g) * torch.where(torch.arange(8) % 2 == 0, 1e-4, 1.0)[:, None]
    gamma, beta = torch.rand(512, generator=g) + 0.5, torch.randn(512, generator=g)
    ref = ln_fwd_ref(z.double(), gamma.double(), beta.double(), 1e-8)[0]
    check_units("fp32 LayerNorm", ln_fwd_ref(z, gamma, beta, 1e-8)[0], ref, F32_RTOL)
    with pytest.raises(AssertionError):
        check_units("LayerNorm with eps 1e-5", ln_fwd_ref(z.double(), gamma.double(), beta.double(), 1e-5)[0], ref,
                    F32_RTOL)


def test_dropout_comparators_reject_one_flipped_mask_bit():
    g = torch.Generator().manual_seed(3)
    M, N = 16, 512
    u = _bf(torch.randn(M, N, dtype=F64, generator=g) * 1.5)
    keep = keep_rows(8, 14, M, N, 0.1)
    ref = _bf(_bf(gelu_ref(u)) * keep)
    check_bf16("fp32 gelu dropout", _bf(_bf(gelu_ref(u.float())).float() * keep.float()), ref)
    bad_keep = keep.clone()
    r = 5
    c = int((gelu_ref(u[r]).abs() * (keep[r] != 0)).argmax())  # the largest kept element of row 5 is dropped
    bad_keep[r, c] = 0.0
    bad = _bf(_bf(gelu_ref(u)) * bad_keep)
    with pytest.raises(AssertionError):
        check_bf16("gelu dropout, one flipped bit", bad, ref)
    with pytest.raises(AssertionError):
        check_exact("zero pattern, one flipped bit", bad == 0, ref == 0)


def test_cross_entropy_comparator_rejects_a_target_shifted_by_one_position():
    g = torch.Generator().manual_seed(4)
    B, T, V, pad = 2, 6, 1000, 0
    tokens = torch.randint(1, V, (B, T), generator=g)
    logits = _bf(torch.randn(B * T, V, dtype=F64, generator=g) * 3)
    _, grad, _, _ = ce_ref(logits, tokens, pad, 1)
    check_bf16("fp32 dlogits", _bf(ce_ref(logits.float(), tokens, pad, 1)[1]), grad)
    bad_tokens = tokens.clone()
    bad_tokens[0, 3] = tokens[0, 4]  # row (0, 2) takes the target of position t + 2
    _, bad, _, _ = ce_ref(logits, bad_tokens, pad, 1)
    with pytest.raises(AssertionError):
        check_bf16("dlogits, one shifted target", _bf(bad), grad)


def test_colsum_comparator_rejects_one_column_left_out():
    g = torch.Generator().manual_seed(5)
    x = _bf(torch.randn(300, 64, dtype=F64, generator=g))
    s, mag = colsum_ref(x)
    check_sum("fp32 column sums", x.float().sum(0), s, mag)
    bad = s.clone()
    bad[17] = 0.0
    with pytest.raises(AssertionError):
        check_sum("column sums, one column left out", bad, s, mag)


def test_argmax_comparator_rejects_the_last_of_tied_maxima():
    x = _argmax_input(255, 264, torch.Generator().manual_seed(6))[:, :255]
    ref = argmax_ref(x)
    last = x.shape[1] - 1 - argmax_ref(x.flip(1))
    with pytest.raises(AssertionError):
        check_exact("argmax taking the last tie", last, ref)


# ------------------------------------------------------------------------------------------------ CPU: argument checks
def _rc(name, *args):
    from virtex_b200 import ops
    return ops._get(name)(*args)


def test_head_entry_points_reject_unsupported_shapes_before_touching_the_device():
    """Each call is invalid only in the one argument named; the library returns VTX_EINVAL (-1) while validating, so
    no pointer (all fake, 256) is dereferenced and no device is needed."""
    P = 256
    # LayerNorm backward: the float4 loops need H % 128 == 0, like the forwards that produce z and stats
    for ln in (1, 0):
        assert _rc("vtx_ln_bwd", P, 0, P, P, P, 0, P, P, P, P, 4, 100, 0.0, 0, 0, ln, 0) == -1
    # attention: at most 32 queries and 64 keys
    assert _rc("vtx_attn_fwd", P, 192, P, 192, P, 192, P, 64, P, 1, 1, 33, 30, P, 1, 0.0, 0, 0, 0) == -1
    assert _rc("vtx_attn_fwd", P, 192, P, 192, P, 192, P, 64, P, 1, 1, 30, 65, P, 1, 0.0, 0, 0, 0) == -1
    assert _rc("vtx_attn_bwd", P, 192, P, 192, P, 192, P, 64, P, P, 64, P, 64, P, 64, 1, 1, 33, 30, P, 1, 0.0, 0, 0,
               0) == -1
    # cross entropy: rows are read 8 logits at a time
    assert _rc("vtx_cross_entropy", P, 1008, P, 1, 30, 1001, 0, 1, P, P, 1, 0) == -1
