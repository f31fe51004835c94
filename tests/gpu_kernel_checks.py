"""Per-kernel parity checks (GPU). Each ``check_*`` returns a dict with error statistics and raises AssertionError
on failure. The checker is plain PyTorch fp32 math (or numpy/scipy for the integer tail; fp64 with a bound derived from
the arithmetic for the attention edge and norm cancellation checks) on the same seeded inputs; the thing under test
always goes through the C ABI (ops.py -> libldmseg_b200.so).

Used by tests/test_kernels_gpu.py (pytest -m gpu) and by tools/gpu_diag.py (one subprocess per check, so a trapped
kernel cannot take the other checks down with it).
"""
import math

import numpy as np
import torch
import torch.nn.functional as F

from video_latent_diffusion_panoptic_segmentation_b200 import _lib as L
from video_latent_diffusion_panoptic_segmentation_b200 import ops

DEV = "cuda"
bf16 = torch.bfloat16


def _poison(t):
    """Outputs start poisoned (NaN / a sentinel), so that an element a kernel fails to write cannot pass by luck."""
    return t.fill_(float("nan")) if t.is_floating_point() else t.fill_(-12345)


def _empty(*a, **k):
    return _poison(torch.empty(*a, **k))


def _empty_like(*a, **k):
    return _poison(torch.empty_like(*a, **k))


def _gen(seed):
    g = torch.Generator(device="cpu")
    g.manual_seed(seed)
    return g


def _randn(shape, seed, scale=1.0, dtype=torch.float32):
    return (torch.randn(shape, generator=_gen(seed)) * scale).to(dtype).to(DEV)


def _stats(got, ref, name, atol, rtol):
    got = got.float()
    ref = ref.float()
    err = (got - ref).abs()
    denom = ref.abs().max().item() + 1e-12
    res = {
        "name": name,
        "max_abs": err.max().item(),
        "ref_max": denom,
        "rel_l2": (err.pow(2).sum().sqrt() / (ref.pow(2).sum().sqrt() + 1e-12)).item(),
        "nan": bool(torch.isnan(got).any().item()),
    }
    bad = err > (atol + rtol * ref.abs())
    res["n_bad"] = int(bad.sum().item())
    res["n"] = got.numel()
    if res["n_bad"] or res["nan"]:
        idx = bad.nonzero()[:8].tolist()
        res["first_bad"] = idx
        raise AssertionError(f"{name}: {res}")
    return res


# ----------------------------------------------------------------------------------------------------------- bound
# Checks against an fp64 reference with a bound derived from the arithmetic instead of atol + rtol |ref|:
#     |got - ref| <= r |ref| + a mag
# mag is the same operation on absolute values (sum_j p_ij |v_j| for attention, |gamma x_hat| + |beta| for the norms):
# it is the scale of the intermediate values, which is what fp32 accumulation and the rounding of intermediates err
# against. r covers the rounding of the output; a covers everything before it. The constants have to satisfy two
# conditions: the kernels stay at or below a quarter of the bound (BOUND_HEADROOM, asserted by the GPU checks), and
# small, plausible bugs in a reference go above it (tests/test_bound_controls.py, on the CPU).
U_BF16 = 2.0 ** -8           # unit roundoff of bf16 (8 significant bits): the rounding of a bf16 output
BOUND_HEADROOM = 0.25
# attention: the bf16 P perturbs the numerator by up to u mag and, at d = 80 / 160 where the row sum stays fp32 (not the
# ones row of the same bf16 P), the quotient by up to u |out| <= u mag: one bf16 ulp, seen on the B200 for constant V.
# MUFU / polynomial ex2 (~1e-4) and fp32 accumulation over <= 7 488 keys are far below u. With the output rounding,
# a correct kernel errs by up to u |ref| + 2u mag <= 3u mag; a = 11u makes the bound at least four times that.
A_ATTN = 11 * U_BF16
# GroupNorm / LayerNorm: GroupNorm takes E[x^2] - mean^2. Its fp32 partial sums are nested sequential sums of a few
# dozen terms per level (a thread's pixels, the pixel lanes, a group's channels, or a warp tree), and only the fold over
# CTAs is fp64. Their relative error eps is ~40 * 2^-24 ~ 2^-19 worst case and ~2^-22 for rounding of random sign.
# The variance carries eps (1 + (mean / spread)^2) / 2 into rstd. For the 64x groups of the cancellation checks, that
# is ~2^-11 typically; the B200 measures ~2^-13 (worst ratio 0.207 against the 0.2 of the output rounding alone). The
# worst case, ~2^-8, would reach the bound. LayerNorm is two-pass (~2^-20). The fp32 affine adds ~2^-23. 4u keeps the
# output rounding under a quarter of the bound, as for attention.
A_NORM = 4 * U_BF16


def bound_ratio(got, ref, mag, r, a):
    """err / (r |ref| + a mag), elementwise in fp64; NaN / inf in `got` (or an error where the bound is 0) give inf."""
    ref = ref.double()
    err = (got.double() - ref).abs()
    ratio = err / (r * ref.abs() + a * mag.double())
    return torch.where(torch.isfinite(err) & ((err == 0) | torch.isfinite(ratio)), ratio.nan_to_num(0.0),
                       torch.full_like(ratio, float("inf")))


def _bound_stats(got, ref, mag, name, r, a, limit=BOUND_HEADROOM, where=None):
    """Raise AssertionError if some element exceeds `limit` x the bound. `where(index)` names a bad element's place in
    the kernel's work decomposition (tile, warp slice, ...)."""
    ratio = bound_ratio(got, ref, mag, r, a)
    worst = ratio.max().item()
    bad = ratio > limit
    res = {"name": name, "worst_ratio": worst, "n_bad": int(bad.sum().item()), "n": ratio.numel(),
           "nan": bool(torch.isnan(got.float()).any().item())}
    if res["n_bad"]:
        idx = tuple(bad.nonzero()[0].tolist())
        res["first_bad"] = idx
        res["first_bad_got_ref_mag"] = (got[idx].item(), ref[idx].item(), mag[idx].item())
        if where is not None:
            res["first_bad_at"] = where(idx)
        raise AssertionError(f"{name}: {res['n_bad']} of {res['n']} elements above {limit} x bound: {res}")
    return res


def attn_ref(q, k, v, scale, qblock=1024):
    """softmax(q k^T * scale) v in fp64, the row maximum subtracted, per (image, head) and per query block (no
    [seq, kv_seq] matrix for all heads at once). q [BH, S, d], k / v [BH, kv_seq, d]: the bf16 values the kernel read.
    Returns (ref, mag), mag = sum_j p_ij |v_j|."""
    BH, S, d = q.shape
    ref = torch.empty((BH, S, d), dtype=torch.float64, device=q.device)
    mag = torch.empty_like(ref)
    for b in range(BH):
        kb, vb = k[b].double(), v[b].double()
        for i0 in range(0, S, qblock):
            s = (q[b, i0:i0 + qblock].double() @ kb.t()) * scale
            p = torch.exp(s - s.max(dim=-1, keepdim=True).values)
            p /= p.sum(dim=-1, keepdim=True)
            ref[b, i0:i0 + qblock] = p @ vb
            mag[b, i0:i0 + qblock] = p @ vb.abs()
    return ref, mag


def norm_ref(x, gamma, beta, eps, groups=None, silu=False):
    """GroupNorm (groups given; x [B, HW, C], groups of C / groups channels over all pixels) or LayerNorm (x [rows, C])
    in fp64, two-pass moments. Returns (ref, mag), mag = |gamma x_hat| + |beta| (SiLU: its slope is below 1.1)."""
    xd = x.double()
    if groups is None:
        mean = xd.mean(-1, keepdim=True)
        var = (xd - mean).pow(2).mean(-1, keepdim=True)
        xh = (xd - mean) / torch.sqrt(var + eps)
    else:
        B, HW, C = xd.shape
        xg = xd.view(B, HW, groups, C // groups)
        mean = xg.mean(dim=(1, 3), keepdim=True)
        var = (xg - mean).pow(2).mean(dim=(1, 3), keepdim=True)
        xh = ((xg - mean) / torch.sqrt(var + eps)).view(B, HW, C)
    g, b = gamma.double(), beta.double()
    y = xh * g + b
    mag = (xh * g).abs() + b.abs()
    if silu:
        y = y * torch.sigmoid(y)
        mag = 1.1 * mag
    return y, mag


# ----------------------------------------------------------------------------------------------------------- DDIM
def check_ddim():
    n = 8 * 4 * 48 * 156
    eps, x = _randn((n,), 1), _randn((n,), 2)
    a_t, a_p = torch.tensor(0.0047), torch.tensor(0.0060)
    coef = torch.stack([(1 - a_t) ** 0.5, a_t ** 0.5, a_p ** 0.5, (1 - a_p) ** 0.5]).float().view(1, 4).to(DEV)
    ti = torch.zeros(1, dtype=torch.int32, device=DEV)
    prev, x0 = _empty_like(x), _empty_like(x)
    ops.ddim_step(eps, x, coef, ti, prev, x0)
    c = coef[0].cpu()
    xc, ec = x.cpu(), eps.cpu()
    x0_ref = (xc - c[0] * ec) / c[1]
    prev_ref = c[2] * x0_ref + c[3] * ec
    assert torch.equal(x0.cpu(), x0_ref), "ddim pred_x0 not bit-exact"
    assert torch.equal(prev.cpu(), prev_ref), "ddim prev_sample not bit-exact"
    return {"name": "ddim", "bit_exact": True}


# ----------------------------------------------------------------------------------------------------------- norms
def check_layernorm(C=640, rows=1000):
    x = _randn((rows, C), 3, dtype=bf16)
    g, b = _randn((C,), 4) * 0.2 + 1, _randn((C,), 5) * 0.1
    out = _empty_like(x)
    ops.layernorm(x, g, b, out, 1e-5)
    ref = F.layer_norm(x.float(), (C,), g, b, 1e-5)
    return _stats(out, ref, f"layernorm C={C}", 2e-2, 1e-2)


def check_groupnorm(c1=320, c2=0, HW=468, B=2, silu=True, eps=1e-5):
    x1 = _randn((B, HW, c1), 6, dtype=bf16) * 1.5 + 0.3
    x2 = (_randn((B, HW, c2), 7, dtype=bf16) * 0.7 - 0.2) if c2 else None
    C = c1 + c2
    g, b = _randn((C,), 8) * 0.2 + 1, _randn((C,), 9) * 0.1
    out = _empty((B, HW, C), dtype=bf16, device=DEV)
    stats = ops.gn_scratch(B, 32, DEV)
    ops.groupnorm(x1, g, b, out, stats, x2=x2, groups=32, eps=eps, silu=silu)
    xin = x1 if x2 is None else torch.cat([x1, x2], dim=-1)
    ref = F.group_norm(xin.float().permute(0, 2, 1), 32, g, b, eps)
    if silu:
        ref = F.silu(ref)
    ref = ref.permute(0, 2, 1)
    return _stats(out, ref, f"groupnorm c1={c1} c2={c2} HW={HW}", 3e-2, 2e-2)


# ----------------------------------------------------------------------------------------------------------- small ops
def check_gemv():
    N, K = 1000, 1280
    w = _randn((N, K), 10, 0.05, bf16)
    x = _randn((K,), 11)
    b1, b2 = _randn((N,), 12), _randn((N,), 13)
    out = _empty(N, device=DEV)
    ops.gemv(w, x, out, b1, b2, silu=True)
    ref = F.silu(w.float() @ x + b1 + b2)
    return _stats(out, ref, "gemv", 1e-3, 1e-3)


def check_timestep_sinusoid():
    half = 160
    exponent = -math.log(10000) * torch.arange(0, half, dtype=torch.float32) / half
    freqs = torch.exp(exponent)
    ts = torch.tensor([999, 979, 19], dtype=torch.int64, device=DEV)
    res = None
    for i in range(3):
        ti = torch.tensor([i], dtype=torch.int32, device=DEV)
        out = _empty(2 * half, device=DEV)
        ops.timestep_sinusoid(ts, ti, freqs.to(DEV), out)
        emb = ts[i].float().cpu() * freqs
        ref = torch.cat([torch.cos(emb), torch.sin(emb)])
        res = _stats(out, ref.to(DEV), f"timestep_sinusoid t={int(ts[i])}", 2e-5, 0)
    return res


def check_conv_small_cin():
    B, h, w, cout = 2, 12, 39, 320
    xt, rgb = _randn((B, 4, h, w), 14), _randn((B, 4, h, w), 15)
    wt, bias = _randn((cout, 8, 3, 3), 16, 0.1), _randn((cout,), 17)
    out = _empty((B, h, w, cout), dtype=bf16, device=DEV)
    ops.conv3x3_small_cin([xt, rgb], ops.pack_small_cin_weight(wt), bias, out, scale=1.0)
    ref = F.conv2d(torch.cat([xt, rgb], 1), wt, bias, padding=1).permute(0, 2, 3, 1)
    r = _stats(out, ref, "conv3x3_small_cin(8->320)", 2e-2, 1e-2)
    z = _randn((B, 4, h, w), 18)
    w2, b2 = _randn((256, 4, 3, 3), 19, 0.1), _randn((256,), 20)
    out2 = _empty((B, h, w, 256), dtype=bf16, device=DEV)
    ops.conv3x3_small_cin([z], ops.pack_small_cin_weight(w2), b2, out2, scale=5.0)
    ref2 = F.conv2d(z * 5.0, w2, b2, padding=1).permute(0, 2, 3, 1)
    _stats(out2, ref2, "conv3x3_small_cin(4->256, scale)", 4e-2, 1e-2)
    return r


def check_conv_out():
    B, h, w, cin = 2, 12, 39, 320
    x = _randn((B, h, w, cin), 21, dtype=bf16)
    wt, bias = _randn((4, cin, 3, 3), 22, 0.05), _randn((4,), 23)
    out = _empty((B, 4, h, w), device=DEV)
    ops.conv_out(x, wt, bias, out)
    ref = F.conv2d(x.float().permute(0, 3, 1, 2), wt, bias, padding=1)
    return _stats(out, ref, "conv_out", 2e-3, 1e-3)


def check_gemm_conv_out_nchw():
    B, h, w, cin = 2, 12, 39, 320
    x = _randn((B, h, w, cin), 21, dtype=bf16)
    wt, bias = _randn((4, cin, 3, 3), 22, 0.05), _randn((4,), 23)
    wp = torch.zeros((8, 9 * cin), device=DEV)
    wp[:4] = wt.permute(0, 2, 3, 1).reshape(4, -1)
    bp = torch.zeros(8, device=DEV)
    bp[:4] = bias
    out = torch.full((B, 4, h, w), float("nan"), device=DEV)
    ops.gemm(x, wp.to(bf16), out, taps=9, bias=bp, flags=L.LDM_GEMM_OUT_NCHW_F32, block_n=32, n_store=4)
    ref = F.conv2d(x.float().permute(0, 3, 1, 2), wp[:4].to(bf16).float().view(4, 3, 3, cin).permute(0, 3, 1, 2), bias,
                   padding=1)
    return _stats(out, ref, "conv_out via implicit GEMM (NCHW f32)", 2e-3, 1e-3)


def check_upsample_im2col():
    B, h, w, C = 2, 6, 20, 64
    x = _randn((B, h, w, C), 24, dtype=bf16)
    out = _empty((B, 12, 39, C), dtype=bf16, device=DEV)
    ops.upsample_nearest(x, out)
    ref = F.interpolate(x.float().permute(0, 3, 1, 2), size=(12, 39), mode="nearest").permute(0, 2, 3, 1)
    assert torch.equal(out.float(), ref), "upsample_nearest (size) mismatch"
    out2 = _empty((B, 12, 40, C), dtype=bf16, device=DEV)
    ops.upsample_nearest(x, out2)
    ref2 = F.interpolate(x.float().permute(0, 3, 1, 2), scale_factor=2.0, mode="nearest").permute(0, 2, 3, 1)
    assert torch.equal(out2.float(), ref2), "upsample_nearest (x2) mismatch"
    x3 = _randn((B, 12, 39, C), 25, dtype=bf16)
    oh, ow = 6, 20
    col = _empty((B * oh * ow, 9 * C), dtype=bf16, device=DEV)
    ops.im2col3x3_s2(x3, col)
    unf = F.unfold(x3.float().permute(0, 3, 1, 2), 3, padding=1, stride=2)  # [B, C*9, L] (c-major, tap-minor)
    unf = unf.view(B, C, 9, oh * ow).permute(0, 3, 2, 1).reshape(B * oh * ow, 9 * C)
    assert torch.equal(col.float(), unf), "im2col3x3_s2 mismatch"
    return {"name": "upsample/im2col", "bit_exact": True}


def check_vae_helpers():
    """Kernels added for the RGB VAE encoder: affine few-channel conv, pad-(0,1) stride-2 im2col, row softmax, planar
    bilinear resize, and the unfused attention chain S = Q K^T -> softmax -> P V built from them."""
    B, h, w, cout = 2, 10, 37, 128
    img = torch.rand((B, 3, h, w), generator=_gen(70)).to(DEV)
    wt, bias = _randn((cout, 3, 3, 3), 71, 0.2), _randn((cout,), 72)
    out = _empty((B, h, w, cout), dtype=bf16, device=DEV)
    ops.conv3x3_small_cin([img], ops.pack_small_cin_weight(wt), bias, out, scale=2.0, shift=-1.0)
    ref = F.conv2d(2. * img - 1., wt, bias, padding=1).permute(0, 2, 3, 1)
    r = _stats(out, ref, "conv3x3_small_cin(3->128, 2x-1)", 2e-2, 1e-2)
    # Downsample2D(padding=0): F.pad(x, (0, 1, 0, 1)) + unfold(stride 2, no padding); even and odd extents
    for (hh, ww) in ((12, 38), (11, 39)):
        C = 64
        x3 = _randn((B, hh, ww, C), 73, dtype=bf16)
        oh, ow = (hh - 2) // 2 + 1, (ww - 2) // 2 + 1
        col = _empty((B * oh * ow, 9 * C), dtype=bf16, device=DEV)
        ops.im2col3x3_s2(x3, col, pad_lo=0)
        unf = F.unfold(F.pad(x3.float().permute(0, 3, 1, 2), (0, 1, 0, 1)), 3, padding=0, stride=2)
        assert unf.shape[-1] == oh * ow
        unf = unf.view(B, C, 9, oh * ow).permute(0, 3, 2, 1).reshape(B * oh * ow, 9 * C)
        assert torch.equal(col.float(), unf), "im2col3x3_s2 pad_lo=0 mismatch"
    # row softmax (vector and scalar paths)
    for (rows, cols) in ((100, 7488), (33, 333)):
        sc = _randn((rows, cols), 74, 6.0)
        pr = _empty((rows, cols), dtype=bf16, device=DEV)
        ops.softmax_rows(sc, pr, 512 ** -0.5)
        ref_p = torch.softmax(sc * 512 ** -0.5, dim=-1)
        _stats(pr, ref_p, f"softmax_rows {rows}x{cols}", 1e-5, 1e-2)
    # planar bilinear resize against F.interpolate (same fp32 formulation)
    xin = _randn((2, 3, 21, 50), 75)
    for size in ((16, 32), (48, 156), (21, 50)):
        o = _empty((2, 3) + size, dtype=torch.float32, device=DEV)
        ops.resize_bilinear_planar(xin, o)
        ref_r = F.interpolate(xin, size=size, mode="bilinear", align_corners=False)
        _stats(o, ref_r, f"resize_bilinear_planar {size}", 2e-6, 1e-6)
    # unfused single-head attention, d = 512: V^T by a role-swapped GEMM, fp32 scores, softmax, P V
    seq, d = 160, 512
    xq, xk, xv = _randn((seq, d), 76, dtype=bf16), _randn((seq, d), 77, dtype=bf16), _randn((seq, d), 78, dtype=bf16)
    wv = _randn((d, d), 79, d ** -0.5, dtype=bf16)
    vt = _empty((d, seq), dtype=bf16, device=DEV)
    ops.gemm(wv, xv, vt)
    sc = _empty((seq, seq), dtype=torch.float32, device=DEV)
    ops.gemm(xq, xk, sc, flags=L.LDM_GEMM_OUT_F32)
    pr = _empty((seq, seq), dtype=bf16, device=DEV)
    ops.softmax_rows(sc, pr, d ** -0.5)
    o = _empty((seq, d), dtype=bf16, device=DEV)
    ops.gemm(pr, vt, o)
    v_ref = xv.float() @ wv.float().t()
    ref_o = torch.softmax(xq.float() @ xk.float().t() * d ** -0.5, dim=-1) @ v_ref
    _stats(vt, v_ref.t(), "V^T by swapped GEMM", 3e-2, 1e-2)
    _stats(o, ref_o, "unfused attention d=512", 3e-2, 2e-2)
    return r


# ----------------------------------------------------------------------------------------------------------- GEMM
def _gemm_ref(a, w, bias=None, residual=None):
    ref = a.float() @ w.float().t()
    if bias is not None:
        ref = ref + bias
    if residual is not None:
        ref = ref + residual.float()
    return ref


def check_gemm_tiny():
    """Smallest possible tcgen05 tile: one k-block, one tile. Prints structure of the error if any."""
    M, N, K = 128, 32, 64
    a = _randn((M, K), 30, 1.0, bf16)
    w = _randn((N, K), 31, 1.0, bf16)
    out = _empty((M, N), dtype=torch.float32, device=DEV)
    ops.gemm(a, w, out, flags=L.LDM_GEMM_OUT_F32, block_n=32)
    torch.cuda.synchronize()
    ref = _gemm_ref(a, w)
    err = (out - ref).abs()
    info = {"name": "gemm_tiny", "max_abs": err.max().item(),
            "rows_bad": int((err.max(dim=1).values > 1e-2).sum()), "cols_bad": int((err.max(dim=0).values > 1e-2).sum())}
    if info["max_abs"] > 1e-2:
        # structural hints for descriptor bugs
        info["out[0,:4]"] = out[0, :4].tolist()
        info["ref[0,:4]"] = ref[0, :4].tolist()
        info["out[1,:4]"] = out[1, :4].tolist()
        info["ref[1,:4]"] = ref[1, :4].tolist()
        # is it the k=0..15 partial product only?
        for kk in (16, 32, 48):
            part = a[:, :kk].float() @ w[:, :kk].float().t()
            info[f"matches_first_{kk}_k"] = bool((out - part).abs().max().item() < 1e-2)
        raise AssertionError(str(info))
    return info


def check_gemm_plain(M=1000, N=320, K=320, block_n=0, bias=True, residual=True, f32out=False):
    a = _randn((M, K), 32, 1.0, bf16)
    w = _randn((N, K), 33, 0.05, bf16)
    b = _randn((N,), 34) if bias else None
    r = _randn((M, N), 35, 1.0, bf16) if residual else None
    out = _empty((M, N), dtype=torch.float32 if f32out else bf16, device=DEV)
    ops.gemm(a, w, out, bias=b, residual=r, flags=L.LDM_GEMM_OUT_F32 if f32out else 0, block_n=block_n)
    ref = _gemm_ref(a, w, b, r)
    return _stats(out, ref, f"gemm M={M} N={N} K={K} bn={block_n}", 3e-2 if not f32out else 2e-3, 1e-2)


def check_gemm_conv3x3(B=2, H=12, W=39, c1=128, c2=0, N=192, block_n=0):
    x1 = _randn((B, H, W, c1), 36, 1.0, bf16)
    x2 = _randn((B, H, W, c2), 37, 1.0, bf16) if c2 else None
    C = c1 + c2
    wt = _randn((N, C, 3, 3), 38, 0.03)
    wp = wt.permute(0, 2, 3, 1).reshape(N, 9 * C).contiguous().to(bf16)
    bias = _randn((N,), 39)
    res = _randn((B * H * W, N), 40, 1.0, bf16)
    out = _empty((B, H, W, N), dtype=bf16, device=DEV)
    ops.gemm(x1, wp, out, a2=x2, taps=9, bias=bias, residual=res, block_n=block_n)
    xin = x1 if x2 is None else torch.cat([x1, x2], -1)
    ref = F.conv2d(xin.float().permute(0, 3, 1, 2), wp.float().view(N, 3, 3, C).permute(0, 3, 1, 2), bias, padding=1)
    ref = ref.permute(0, 2, 3, 1) + res.float().view(B, H, W, N)
    return _stats(out, ref, f"conv3x3 B={B} {H}x{W} c1={c1} c2={c2} N={N}", 5e-2, 2e-2)


def check_gemm_conv3x3_stride2(B=2, H=24, W=78, c1=128, N=192, pad=1, silu=False):
    """Conv2d(3x3, stride 2) as an implicit GEMM through element-strided tensor maps (ldm_gemm_desc.a_stride), padding 1
    (diffusers Downsample2D of the UNet, the seg-AE encoder) and F.pad(0, 1, 0, 1) + padding 0 (the RGB VAE's)."""
    x = _randn((B, H, W, c1), 136, 1.0, bf16)
    wt = _randn((N, c1, 3, 3), 138, 0.03)
    wp = wt.permute(0, 2, 3, 1).reshape(N, 9 * c1).contiguous().to(bf16)
    bias = _randn((N,), 139)
    xin = x.float().permute(0, 3, 1, 2)
    if pad == 0:
        xin = F.pad(xin, (0, 1, 0, 1))
    ref = F.conv2d(xin, wp.float().view(N, 3, 3, c1).permute(0, 3, 1, 2), bias, stride=2, padding=pad)
    if silu:
        ref = F.silu(ref)
    oh, ow = ref.shape[-2:]
    out = _empty((B, oh, ow, N), dtype=bf16, device=DEV)
    ops.gemm(x, wp, out, taps=9, bias=bias, a_stride=2, a_pad=pad, flags=L.LDM_GEMM_SILU if silu else 0)
    return _stats(out, ref.permute(0, 2, 3, 1), f"conv3x3 stride 2 pad={pad} B={B} {H}x{W} -> {oh}x{ow} c={c1} N={N}",
                  5e-2, 2e-2)


def check_gemm_upsample_conv3x3(B=2, H=12, W=39, C=128, N=128):
    """F.interpolate(scale 2, nearest) + Conv2d(3x3, padding 1) as four 2x2 convolutions of the low-resolution input
    written through an element-strided output map (ldm_gemm_desc.up2). Reference: the two torch ops on the bf16 input
    with the ORIGINAL 3x3 weights rounded to bf16 (what the gather-pass path computes)."""
    x = _randn((B, H, W, C), 146, 1.0, bf16)
    wt = _randn((N, 3, 3, C), 148, 0.03)
    bias = _randn((N,), 149)
    w4, b4 = ops.fold_upsample_conv3x3(wt, bias)
    out = _empty((B, 2 * H, 2 * W, N), dtype=bf16, device=DEV)
    ops.gemm(x, w4, out, taps=4, bias=b4, up2=True)
    up = F.interpolate(x.float().permute(0, 3, 1, 2), scale_factor=2, mode="nearest")
    ref = F.conv2d(up, wt.to(bf16).float().permute(0, 3, 1, 2), bias, padding=1).permute(0, 2, 3, 1)
    # and the path it replaces, on the same inputs: the collapsed kernel must not be further from fp32 than it is
    upb = _empty((B, 2 * H, 2 * W, C), dtype=bf16, device=DEV)
    ops.upsample_nearest(x, upb)
    out2 = _empty((B, 2 * H, 2 * W, N), dtype=bf16, device=DEV)
    ops.gemm(upb, wt.reshape(N, 9 * C).to(bf16).contiguous(), out2, taps=9, bias=bias)
    ref32 = F.conv2d(up, wt.permute(0, 3, 1, 2), bias, padding=1).permute(0, 2, 3, 1)
    rel = lambda o: ((o.float() - ref32).pow(2).sum().sqrt() / ref32.pow(2).sum().sqrt()).item()
    assert rel(out) <= 1.5 * rel(out2) + 1e-3, f"up2 rel L2 {rel(out):.2e} vs gather path {rel(out2):.2e}"
    r = _stats(out, ref, f"upsample x2 + conv3x3 B={B} {H}x{W} C={C} N={N}", 6e-2, 2e-2)
    r["rel_l2_gather_path"] = rel(out2)
    r["rel_l2_fp32_weights"] = rel(out)
    return r


def check_gemm_splitk(B=1, H=6, W=20, c1=1280, c2=0, N=1280, taps=9, residual=True, rowbias=True):
    """Long K, few tiles: the K range of every tile is cut into work items (ldm_gemm_desc.splitk_ws); the partials are
    added in slice order by a second small launch, so repeated launches are bit-identical."""
    x1 = _randn((B, H, W, c1), 36, 1.0, bf16)
    x2 = _randn((B, H, W, c2), 37, 1.0, bf16) if c2 else None
    C = c1 + c2
    wp = _randn((N, taps * C), 38, 0.01, bf16)
    bias = _randn((N,), 39)
    rb = _randn((B, N), 41) if rowbias else None
    res = _randn((B * H * W, N), 40, 1.0, bf16) if residual else None
    outs = []
    for _ in range(3):
        out = _empty((B, H, W, N), dtype=bf16, device=DEV)
        ops.gemm(x1, wp, out, a2=x2, taps=taps, bias=bias, rowbias=rb, residual=res)
        outs.append(out)
    bn, pair, split = ops.gemm_last_config()
    assert split > 1, f"expected a split-K launch for M={B * H * W} K={taps * C}, got block_n={bn} pair={pair} split={split}"
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2]), "split-K launches are not bit-reproducible"
    xin = x1 if x2 is None else torch.cat([x1, x2], -1)
    if taps == 9:
        ref = F.conv2d(xin.float().permute(0, 3, 1, 2), wp.float().view(N, 3, 3, C).permute(0, 3, 1, 2), bias, padding=1)
        ref = ref.permute(0, 2, 3, 1)
    else:
        ref = xin.float() @ wp.float().t() + bias
    if rowbias:
        ref = ref + rb.view(B, 1, 1, N)
    if residual:
        ref = ref + res.float().view(B, H, W, N)
    return _stats(outs[0], ref, f"split-K x{split} bn={bn} pair={pair} B={B} {H}x{W} C={C} N={N} taps={taps}", 5e-2, 2e-2)


def check_gemm_concat_1x1():
    B, H, W, c1, c2, N = 2, 6, 20, 128, 64, 128
    x1, x2 = _randn((B, H, W, c1), 41, 1.0, bf16), _randn((B, H, W, c2), 42, 1.0, bf16)
    w = _randn((N, c1 + c2), 43, 0.05, bf16)
    bias = _randn((N,), 44)
    out = _empty((B, H, W, N), dtype=bf16, device=DEV)
    ops.gemm(x1, w, out, a2=x2, taps=1, bias=bias)
    ref = torch.cat([x1, x2], -1).float() @ w.float().t() + bias
    return _stats(out, ref, "conv1x1 concat", 3e-2, 1e-2)


def check_gemm_geglu():
    M, C = 500, 320
    a = _randn((M, C), 45, 1.0, bf16)
    w = _randn((8 * C, C), 46, 0.05)
    b = _randn((8 * C,), 47)
    inner = 4 * C
    # interleave value/gate rows in blocks of 16 (what the host packer does)
    idx = torch.arange(inner).view(-1, 16)
    perm = torch.cat([idx, idx + inner], dim=1).reshape(-1).to(DEV)
    wp, bp = w[perm].contiguous().to(bf16), b[perm].contiguous()
    out = _empty((M, inner), dtype=bf16, device=DEV)
    ops.gemm(a, wp, out, bias=bp, flags=L.LDM_GEMM_GEGLU)
    h = a.float() @ w.to(bf16).float().t() + b
    val, gate = h.chunk(2, dim=-1)
    ref = val * F.gelu(gate)
    return _stats(out, ref, "gemm GEGLU", 3e-2, 2e-2)


def check_ln_fold(kind="qkv", B=2, heads=8, d=40, seq=300, mean_shift=0.5):
    """LayerNorm folded into the GEMMs around it (ldm_gemm_desc.ln_stats): the producer GEMM (bias + residual) writes
    the per-row moments of its bf16 output; the consumer (QKV split or GEGLU) runs on the raw rows with gamma-scaled
    weights and normalises in its epilogue. Reference: fp32 LayerNorm of the producer's bf16 output, then the Linear."""
    C = heads * d
    M = B * seq
    a = _randn((M, C), 90, 1.0, bf16)
    wprod = _randn((C, C), 91, 0.05, bf16)
    bprod = _randn((C,), 92) + mean_shift          # a row mean that is not small against the spread
    res = _randn((M, C), 93, 1.0, bf16)
    x = _empty((M, C), dtype=bf16, device=DEV)
    stats = _empty(((C + 31) // 32, M, 2), dtype=torch.float32, device=DEV)   # part-major
    stats.fill_(float("nan"))
    ops.gemm(a, wprod, x, bias=bprod, residual=res, row_stats=stats)
    xs = x.float().view(M, -1, 32).transpose(0, 1)
    assert not torch.isnan(stats).any(), "row_stats has unwritten entries"
    _stats(stats[:, :, 0], xs.sum(-1), "row_stats sum", 2e-3, 1e-4)
    _stats(stats[:, :, 1], xs.pow(2).sum(-1), "row_stats sum of squares", 2e-3, 1e-4)
    gamma, beta = _randn((C,), 94) * 0.3 + 1.0, _randn((C,), 95) * 0.2
    xn = F.layer_norm(x.float(), (C,), gamma, beta, 1e-5)
    if kind == "qkv":
        w = _randn((3 * C, C), 96, 0.05)
        w2, b2, colsum = ops.fold_layernorm(w, None, gamma, beta)
        q, k, vt, dpad, seq_pad = _alloc_qkv(B, heads, seq, d)
        ops.gemm(x, w2, None, bias=b2, flags=L.LDM_GEMM_QKV_SPLIT, ln_fold=(stats, colsum, 1e-5),
                 qkv=dict(q=q, k=k, vt=vt, heads=heads, head_dim=d, dpad=dpad, seq=seq, seq_pad=seq_pad))
        ref = (xn @ w.t()).view(B, seq, 3, heads, d)
        qr = ref[:, :, 0].permute(0, 2, 1, 3).reshape(B * heads, seq, d)
        kr = ref[:, :, 1].permute(0, 2, 1, 3).reshape(B * heads, seq, d)
        vr = ref[:, :, 2].permute(0, 2, 3, 1).reshape(B * heads, d, seq)
        _stats(q[:, :, :d], qr, "ln-fold qkv q", 4e-2, 2e-2)
        _stats(k[:, :, :d], kr, "ln-fold qkv k", 4e-2, 2e-2)
        assert float(q[:, :, d:].abs().max()) == 0.0, "q padding overwritten"
        return _stats(vt[:, :d, :seq], vr, f"ln-fold qkv vt d={d} seq={seq}", 4e-2, 2e-2)
    inner = 4 * C
    w, b = _randn((8 * C, C), 97, 0.05), _randn((8 * C,), 98)
    idx = torch.arange(inner).view(-1, 16)
    perm = torch.cat([idx, idx + inner], dim=1).reshape(-1).to(DEV)
    w2, b2, colsum = ops.fold_layernorm(w[perm].contiguous(), b[perm].contiguous(), gamma, beta)
    out = _empty((M, inner), dtype=bf16, device=DEV)
    ops.gemm(x, w2, out, bias=b2, flags=L.LDM_GEMM_GEGLU, ln_fold=(stats, colsum, 1e-5))
    val, gate = (xn @ w.t() + b).chunk(2, dim=-1)
    ref = val * F.gelu(gate)
    # the un-folded path on the same inputs (LayerNorm kernel -> bf16 -> GEMM): the fold must not be less accurate
    xl, out2 = _empty((M, C), dtype=bf16, device=DEV), _empty((M, inner), dtype=bf16, device=DEV)
    ops.layernorm(x, gamma, beta, xl, 1e-5)
    ops.gemm(xl, w[perm].contiguous().to(bf16), out2, bias=b[perm].contiguous(), flags=L.LDM_GEMM_GEGLU)
    rel = lambda o: ((o.float() - ref).pow(2).sum().sqrt() / ref.pow(2).sum().sqrt()).item()
    assert rel(out) <= 1.25 * rel(out2) + 5e-4, f"ln-fold GEGLU rel L2 {rel(out):.2e} vs un-folded {rel(out2):.2e}"
    r = _stats(out, ref, f"ln-fold GEGLU C={C} M={M}", 8e-2, 3e-2)
    r["rel_l2_unfolded"] = rel(out2)
    return r


def _alloc_qkv(B, heads, seq, d):
    q = ops.alloc_qkv(B, heads, seq, d, DEV)
    return q["q"], q["k"], q["vt"], q["dpad"], q["seq_pad"]


def check_gemm_qkv(B=2, heads=8, d=40, seq=300):
    C = heads * d
    a = _randn((B * seq, C), 48, 1.0, bf16)
    w = _randn((3 * C, C), 49, 0.05, bf16)
    q, k, vt, dpad, seq_pad = _alloc_qkv(B, heads, seq, d)
    ops.gemm(a, w, None, flags=L.LDM_GEMM_QKV_SPLIT,
             qkv=dict(q=q, k=k, vt=vt, heads=heads, head_dim=d, dpad=dpad, seq=seq, seq_pad=seq_pad))
    ref = (a.float() @ w.float().t()).view(B, seq, 3, heads, d)
    qr = ref[:, :, 0].permute(0, 2, 1, 3).reshape(B * heads, seq, d)
    kr = ref[:, :, 1].permute(0, 2, 1, 3).reshape(B * heads, seq, d)
    vr = ref[:, :, 2].permute(0, 2, 3, 1).reshape(B * heads, d, seq)
    if vt.shape[1] != d:  # ones row (softmax row sums come out of the PV MMA) + zero rows must be untouched
        assert float((vt[:, d, :seq] - 1).abs().max()) == 0.0 and float(vt[:, d + 1:].abs().max()) == 0.0
    _stats(q[:, :, :d], qr, "qkv q", 3e-2, 1e-2)
    _stats(k[:, :, :d], kr, "qkv k", 3e-2, 1e-2)
    assert float(q[:, :, d:].abs().max()) == 0.0, "q padding overwritten"
    return _stats(vt[:, :d, :seq], vr, f"qkv vt d={d}", 3e-2, 1e-2)


def check_gemm_convt():
    B, H, W, cin, cout = 2, 6, 20, 256, 256
    x = _randn((B, H, W, cin), 50, 1.0, bf16)
    wt = _randn((cin, cout, 2, 2), 51, 0.05)
    bias = _randn((cout,), 52)
    g, be = _randn((cout,), 53) * 0.2 + 1, _randn((cout,), 54) * 0.1
    wp = wt.permute(2, 3, 1, 0).reshape(4 * cout, cin).contiguous().to(bf16)  # [(dy,dx,co), ci]
    bp = bias.repeat(4).contiguous()
    out = _empty((B, 2 * H, 2 * W, cout), dtype=bf16, device=DEV)
    ops.gemm(x, wp, out, bias=bp, flags=L.LDM_GEMM_CONVT_LN_SILU, block_n=cout, ln=(g, be, 1e-6))
    wq = wp.float().view(2, 2, cout, cin).permute(3, 2, 0, 1)
    y = F.conv_transpose2d(x.float().permute(0, 3, 1, 2), wq, bias, stride=2)
    u = y.mean(1, keepdim=True)
    s = (y - u).pow(2).mean(1, keepdim=True)
    y = (y - u) / torch.sqrt(s + 1e-6)
    y = F.silu(g[:, None, None] * y + be[:, None, None]).permute(0, 2, 3, 1)
    return _stats(out, y, "convT+LN2d+SiLU", 4e-2, 2e-2)


# ----------------------------------------------------------------------------------------------------------- attention
def check_attention(B=1, heads=2, d=40, seq=300, log2_units=False, spread=1.0):
    """log2_units: q arrives pre-multiplied by d^-0.5 * log2(e) (as the UNet's packed QKV weight produces it) and the
    kernel is told scale = ln 2; spread > 1 widens the score range (running maxima that keep growing, lazy rescales)."""
    q, k, vt, dpad, seq_pad = _alloc_qkv(B, heads, seq, d)
    qf = _randn((B * heads, seq, d), 55, spread, bf16)
    kf = _randn((B * heads, seq, d), 56, 1.0, bf16)
    vf = _randn((B * heads, seq, d), 57, 1.0, bf16)
    q[:, :, :d] = qf
    k[:, :, :d] = kf
    vt[:, :d, :seq] = vf.transpose(1, 2)
    out = _empty((B * seq, heads * d), dtype=bf16, device=DEV)
    if log2_units:
        import math
        qs = (qf.float() * (d ** -0.5 * math.log2(math.e))).to(bf16)
        q[:, :, :d] = qs
        ops.flash_attn(q, k, vt, out, B=B, heads=heads, seq=seq, head_dim=d, dpad=dpad, seq_pad=seq_pad,
                       scale=math.log(2.0))
        ref = F.scaled_dot_product_attention(qs.float(), kf.float(), vf.float(), scale=math.log(2.0))
    else:
        ops.flash_attn(q, k, vt, out, B=B, heads=heads, seq=seq, head_dim=d, dpad=dpad, seq_pad=seq_pad, scale=d ** -0.5)
        ref = F.scaled_dot_product_attention(qf.float(), kf.float(), vf.float())  # [BH, seq, d]
    ref = ref.view(B, heads, seq, d).permute(0, 2, 1, 3).reshape(B * seq, heads * d)
    return _stats(out, ref, f"flash_attn d={d} seq={seq} log2_units={log2_units} spread={spread}", 2e-2, 2e-2)


def check_cross_attention(B=2, heads=8, d=40, seq=300, kv_seq=77, ctx_dim=768):
    """attn2 of BasicTransformerBlock built from the C-ABI pieces: to_q through the head-split epilogue (q only),
    to_k | to_v of the context rows through the same epilogue with part0 = 1, flash attention with kv_seq keys."""
    C = heads * d
    x = _randn((B * seq, C), 80, 1.0, bf16)
    ctx = _randn((B * kv_seq, ctx_dim), 81, 1.0, bf16)
    wq = _randn((C, C), 82, C ** -0.5, bf16)
    wkv = _randn((2 * C, ctx_dim), 83, ctx_dim ** -0.5, bf16)
    qb = ops.alloc_qkv(B, heads, seq, d, DEV)
    kv = ops.alloc_kv(B, heads, kv_seq, d, DEV)
    _poison(qb["q"][:, :, :d])
    _poison(kv["k"][:, :, :d])
    _poison(kv["vt"][:, :d, :kv_seq])
    ops.gemm(x, wq, None, flags=L.LDM_GEMM_QKV_SPLIT,
             qkv=dict(q=qb["q"], heads=heads, head_dim=d, dpad=qb["dpad"], seq=seq, seq_pad=qb["seq_pad"]))
    ops.gemm(ctx, wkv, None, flags=L.LDM_GEMM_QKV_SPLIT, qkv=dict(kv, part0=1))
    out = _empty((B * seq, C), dtype=bf16, device=DEV)
    ops.flash_attn(qb["q"], kv["k"], kv["vt"], out, B=B, heads=heads, seq=seq, head_dim=d, dpad=kv["dpad"],
                   seq_pad=kv["seq_pad"], scale=d ** -0.5, kv_seq=kv_seq)
    qr = (x.float() @ wq.float().t()).view(B, seq, heads, d).permute(0, 2, 1, 3)
    kvr = (ctx.float() @ wkv.float().t()).view(B, kv_seq, 2, heads, d)
    kr, vr = kvr[:, :, 0].permute(0, 2, 1, 3), kvr[:, :, 1].permute(0, 2, 1, 3)
    _stats(qb["q"][:, :, :d], qr.reshape(B * heads, seq, d), "cross q", 3e-2, 1e-2)
    _stats(kv["k"][:, :, :d], kr.reshape(B * heads, kv_seq, d), "cross k", 3e-2, 1e-2)
    _stats(kv["vt"][:, :d, :kv_seq], vr.transpose(-1, -2).reshape(B * heads, d, kv_seq), "cross vt", 3e-2, 1e-2)
    if kv["vt"].shape[1] != d:
        assert float((kv["vt"][:, d, :kv_seq] - 1).abs().max()) == 0.0, "ones row of the context V^T overwritten"
    # the checker uses the bf16-rounded projections the kernel saw
    ref = F.scaled_dot_product_attention(qb["q"][:, :, :d].float().view(B, heads, seq, d),
                                         kv["k"][:, :, :d].float().view(B, heads, kv_seq, d),
                                         kv["vt"][:, :d, :kv_seq].float().transpose(1, 2).view(B, heads, kv_seq, d))
    ref = ref.permute(0, 2, 1, 3).reshape(B * seq, C)
    return _stats(out, ref, f"cross attention d={d} seq={seq} kv={kv_seq}", 2e-2, 2e-2)


# ----------------------------------------------------------------------------------------------------------- attention edges
# Inputs chosen so that the data reaches what random scores never do: one dominant key per row at block and half-block
# boundaries, block maxima that jump by more than the lazy (2^8) and redo (2^64) thresholds, rows whose scores all lie
# far below zero or are all equal. fp64 reference with the maximum subtracted (attn_ref), bound comparator above.
LOG2E = math.log2(math.e)
EDGE_KV = (1, 16, 47, 48, 49, 95, 96, 97, 129, 7488)
CROSS_QUERIES = 300   # two 256-query CTAs of the 40-wide kernel, three 128-query tiles of the others, ragged


def _attn_where(idx):
    bh, row, ch = idx
    return {"image_head": bh, "query_row": row, "channel": ch, "query_tile_128": row // 128,
            "warp_slice_32": (row % 128) // 32}


def _attn_launch(q, k, v, d, scale, cross):
    """flash_attn on q [heads, S, d], k / v [heads, kv, d] (bf16, one image): self-attention (S == kv) through one set of
    head-split buffers, cross-attention through a separate key / value set. Returns out [heads, S, d]."""
    heads, S, _ = q.shape
    kv = k.shape[1]
    qb = ops.alloc_qkv(1, heads, S, d, DEV)
    kb = ops.alloc_kv(1, heads, kv, d, DEV) if cross else qb
    assert cross or kv == S
    qb["q"][:, :, :d] = q
    kb["k"][:, :, :d] = k
    kb["vt"][:, :d, :kv] = v.transpose(1, 2)
    out = _empty((S, heads * d), dtype=bf16, device=DEV)
    ops.flash_attn(qb["q"], kb["k"], kb["vt"], out, B=1, heads=heads, seq=S, head_dim=d, dpad=kb["dpad"],
                   seq_pad=kb["seq_pad"], scale=scale, kv_seq=kv if cross else 0)
    return out.view(S, heads, d).transpose(0, 1)


def _bf16_scalar(x):
    return float(torch.tensor(x).to(bf16))


def needle_positions(kv):
    """Key 0, the last key, both sides of the 48-key halves of the 40-wide kernel and of the 64- / 96-key block
    boundaries, and both sides of the start of the ragged last block."""
    pos = {0, kv - 1, 47, 48, 63, 64, 95, 96, 127, 128, 191, 192}
    for blk in (64, 96):
        last = (kv - 1) // blk * blk
        pos |= {last - 1, last}
    return sorted(p for p in pos if 0 <= p < kv)


def needle_inputs(S, kv, d, margin, heads=2, seed=0):
    """Row i of head h attends to key needle_positions(kv)[(i + h) % n]. Key j carries the bits of j as signs in its
    first `bits` channels, the query the needle's signs times sigma: the needle scores sigma * bits, every other key at
    least 2 sigma less, i.e. `margin` log2 units at scale d^-0.5. |V| in [1, 2). Returns q, k, v (bf16) and the needle
    index of every (head, row)."""
    g = _gen(seed)
    bits = max(1, (kv - 1).bit_length())
    assert bits <= d
    scale = d ** -0.5
    sigma = _bf16_scalar(margin / (2 * scale * LOG2E))
    sign = ((torch.arange(kv)[:, None] >> torch.arange(bits)) & 1).float() * 2 - 1      # [kv, bits]
    pos = torch.tensor(needle_positions(kv))
    tgt = pos[(torch.arange(S)[None, :] + torch.arange(heads)[:, None]) % len(pos)]      # [heads, S]
    q = torch.zeros((heads, S, d))
    q[:, :, :bits] = sigma * sign[tgt]
    k = torch.zeros((heads, kv, d))
    k[:, :, :bits] = sign
    v = torch.where(torch.rand((heads, kv, d), generator=g) < 0.5, -1.0, 1.0) * (1 + torch.rand((heads, kv, d), generator=g))
    return q.to(bf16), k.to(bf16), v.to(bf16), tgt


def check_attn_needles(d, cross):
    """Needles on every boundary, margins of 7, 20, 40 and 100 log2 units. With the needle in a block j > 0, that
    block's maximum exceeds the running reference by the margin when an earlier key is one sign flip away (needle 96,
    key 32: the first block of every kernel, the same half in the 40-wide one): at 7, P up to 2^7 accumulates into O without a rescale (the lazy
    threshold is 2^8); at 20 and 40, O is rescaled lazily; at 100, the block's exponentials are redone (> 2^64). From
    20 up, the other keys weigh <= 13 * 2^-20, and the output must be the needle's V row to bf16 rounding."""
    worst = 0.0
    scale = d ** -0.5
    for kv in EDGE_KV:
        S = CROSS_QUERIES if cross else kv
        for margin in (7.0, 20.0, 40.0, 100.0):
            q, k, v, tgt = needle_inputs(S, kv, d, margin, seed=kv)
            q, k, v = q.to(DEV), k.to(DEV), v.to(DEV)
            out = _attn_launch(q, k, v, d, scale, cross)
            ref, mag = attn_ref(q, k, v, scale)
            name = f"attn needles d={d} {'cross' if cross else 'self'} S={S} kv={kv} margin={margin}"
            worst = max(worst, _bound_stats(out, ref, mag, name, U_BF16, A_ATTN, where=_attn_where)["worst_ratio"])
            if margin < 20:
                continue
            want = torch.gather(v, 1, tgt.to(DEV)[:, :, None].expand(-1, -1, d)).float()
            off = (out.float() - want).abs() > U_BF16 * want.abs()
            assert not off.any(), f"{name}: {int(off.sum())} outputs differ from the needle's V row by more than bf16 " \
                                  f"rounding, first at {_attn_where(tuple(off.nonzero()[0].tolist()))}"
    return {"name": f"attn needles d={d} cross={cross}", "worst_ratio": worst}


def check_attn_const_v(d, cross):
    """V constant along the keys: the output must be that constant to one bf16 ulp for any P, i.e. the numerator and the
    row sum (the ones row of V^T at d = 40) see the same P. Peaked random scores (std ~6 log2 units)."""
    worst = 0.0
    scale = d ** -0.5
    for kv in EDGE_KV:
        S = CROSS_QUERIES if cross else kv
        g = _gen(100 + kv)
        q = (torch.randn((2, S, d), generator=g) * 4).to(bf16).to(DEV)
        k = torch.randn((2, kv, d), generator=g).to(bf16).to(DEV)
        c = (torch.where(torch.rand((2, 1, d), generator=g) < 0.5, -1.0, 1.0) *
             (0.5 + 1.5 * torch.rand((2, 1, d), generator=g))).to(bf16).to(DEV)
        v = c.expand(-1, kv, -1).contiguous()
        out = _attn_launch(q, k, v, d, scale, cross)
        ref, mag = attn_ref(q, k, v, scale)
        name = f"attn constant V d={d} {'cross' if cross else 'self'} S={S} kv={kv}"
        worst = max(worst, _bound_stats(out, ref, mag, name, U_BF16, A_ATTN, where=_attn_where)["worst_ratio"])
        ulp = torch.exp2(torch.floor(torch.log2(c.float().abs())) - 7)
        off = (out.float() - c.float()).abs() > ulp
        assert not off.any(), f"{name}: {int(off.sum())} outputs more than one bf16 ulp from the constant, first at " \
                              f"{_attn_where(tuple(off.nonzero()[0].tolist()))}"
    return {"name": f"attn constant V d={d} cross={cross}", "worst_ratio": worst}


def check_attn_flat(d, cross):
    """Every score of a row far below zero (a common offset of -100 / -200 log2 units on scores of std ~1.4), and every
    score of a row equal (all keys the same). Outputs finite and within the bound."""
    worst = 0.0
    scale = d ** -0.5
    for kv in (1, 16, 47, 48, 49, 95, 96, 97, 300):
        S = CROSS_QUERIES if cross else kv
        for case in (-100.0, -200.0, "equal"):
            g = _gen(200 + kv)
            q = torch.randn((2, S, d), generator=g)
            k = torch.randn((2, kv, d), generator=g)
            if case == "equal":
                k = k[:, :1].expand(-1, kv, -1)
            else:   # one channel carries the offset: 8 * kb * scale * log2(e) = offset
                q[:, :, d - 1] = 8.0
                k[:, :, d - 1] = _bf16_scalar(case / (8.0 * scale * LOG2E))
            q, k = q.to(bf16).to(DEV), k.contiguous().to(bf16).to(DEV)
            v = torch.randn((2, kv, d), generator=g).to(bf16).to(DEV)
            out = _attn_launch(q, k, v, d, scale, cross)
            ref, mag = attn_ref(q, k, v, scale)
            name = f"attn flat scores d={d} {'cross' if cross else 'self'} S={S} kv={kv} case={case}"
            worst = max(worst, _bound_stats(out, ref, mag, name, U_BF16, A_ATTN, where=_attn_where)["worst_ratio"])
    return {"name": f"attn flat scores d={d} cross={cross}", "worst_ratio": worst}


def attn_random_inputs(S, kv, d, heads, spread, seed):
    """q ~ N(0, spread^2), k, v ~ N(0, 1) in bf16: scores of std spread * log2(e) log2 units at scale d^-0.5."""
    g = _gen(seed)
    return tuple(torch.randn((heads, n, d), generator=g).mul(s).to(bf16)
                 for n, s in ((S, spread), (kv, 1.0), (kv, 1.0)))


def check_attention_bound(d, seq, heads=2, spread=4.0):
    """Random self-attention against the fp64 reference with the bound comparator, at the largest shape of the plans
    (d = 40, 7 488 tokens): the data tests/test_bound_controls.py shows the comparator's sensitivity on."""
    q, k, v = (t.to(DEV) for t in attn_random_inputs(seq, seq, d, heads, spread, 300 + d))
    out = _attn_launch(q, k, v, d, d ** -0.5, False)
    ref, mag = attn_ref(q, k, v, d ** -0.5)
    return _bound_stats(out, ref, mag, f"attn bound d={d} seq={seq} spread={spread}", U_BF16, A_ATTN, where=_attn_where)


# ----------------------------------------------------------------------------------------------------------- norm cancellation
def cancellation_input(shape, seed):
    """x [n, m, groups, cpg]: every (n, group) has a mean of 16, 32 or 64 times its spread (cycling over the groups,
    random sign), spread in [0.5, 2). In bf16 the 64x groups still resolve spread / 2."""
    n, m, groups, cpg = shape
    g = _gen(seed)
    spread = 0.5 + 1.5 * torch.rand((n, 1, groups, 1), generator=g)
    ratio = torch.tensor([16.0, 32.0, 64.0]).repeat(groups)[:groups].view(1, 1, groups, 1)
    sign = torch.where(torch.rand((n, 1, groups, 1), generator=g) < 0.5, -1.0, 1.0)
    return ((sign * ratio + torch.randn(shape, generator=g)) * spread).to(bf16)


def _kernel_events(fn):
    """torch.profiler events (CUDA activity only) of what `fn` launches. A capture that is not the first of the process
    can lose the record of its first kernel (seen on the B200 after the plan walk's captures): two throw-away kernels
    go first, so that the loss falls on them."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(2):
            torch.zeros(1, device=DEV).add_(1)
            torch.cuda.synchronize()
        fn()
        torch.cuda.synchronize()
    return list(prof.events())


def _launched_kernels(fn):
    """Names of the CUDA kernels `fn` launches."""
    return {e.name for e in _kernel_events(fn)}


GN_KERNELS = ("gn_fused_kernel", "gn_cluster_kernel", "gn_stats_kernel")


def check_groupnorm_cancel(c1, c2, HW, B, silu, kernel, eps=1e-5):
    """`kernel`: the GroupNorm kernel the shape must select (gn_fused_kernel, the cooperative two-sweep kernel, or
    gn_cluster_kernel), so that a change of the selection cannot move this coverage silently."""
    C = c1 + c2
    x = cancellation_input((B, HW, 32, C // 32), 60 + B).view(B, HW, C).to(DEV)
    x1 = x[..., :c1].contiguous()
    x2 = x[..., c1:].contiguous() if c2 else None
    g, b = _randn((C,), 8) * 0.2 + 1, _randn((C,), 9) * 0.1
    out = _empty((B, HW, C), dtype=bf16, device=DEV)
    stats = ops.gn_scratch(B, 32, DEV)
    names = _launched_kernels(lambda: ops.groupnorm(x1, g, b, out, stats, x2=x2, groups=32, eps=eps, silu=silu))
    ran = [k for k in GN_KERNELS if any(k in n for n in names)]
    assert ran == [kernel], f"groupnorm B={B} HW={HW} C={C}: expected {kernel}, launched {ran} ({sorted(names)})"
    assert int(stats[-2 * B:].view(torch.int32).abs().sum()) == 0, "groupnorm left its barrier counters non-zero"
    ref, mag = norm_ref(x, g, b, eps, groups=32, silu=silu)
    return _bound_stats(out, ref, mag, f"groupnorm cancellation c1={c1} c2={c2} HW={HW} B={B} silu={silu}", U_BF16,
                        A_NORM, where=lambda i: {"image": i[0], "pixel": i[1], "group": i[2] // (C // 32)})


def check_layernorm_cancel(C, rows):
    x = cancellation_input((rows, 1, 1, C), 70 + C).view(rows, C).to(DEV)
    g, b = _randn((C,), 4) * 0.2 + 1, _randn((C,), 5) * 0.1
    out = _empty_like(x)
    ops.layernorm(x, g, b, out, 1e-5)
    ref, mag = norm_ref(x, g, b, 1e-5)
    return _bound_stats(out, ref, mag, f"layernorm cancellation C={C} rows={rows}", U_BF16, A_NORM)


# ----------------------------------------------------------------------------------------------------------- integer tail
def check_logits_to_ids(up=2):
    B, h, w, C = 2, 24, 78, 128
    lg = _randn((B, h, w, C), 58, 2.0)
    lg[:, :, :, 5] += 3.0  # a dominant class so that the threshold keeps some pixels
    lg[0, 3, 4, 7] = lg[0, 3, 4, 9] = 50.0  # exact tie -> first index
    H, W = h * up, w * up
    ids = _empty((B, H, W), dtype=torch.int32, device=DEV)
    counts = _empty((B, 2, C), dtype=torch.int32, device=DEV)
    ops.logits_to_ids(lg, ids, counts, up=up, mask_th=0.5, ignore_label=127)
    x = lg.permute(0, 3, 1, 2).cpu()
    if up != 1:
        x = F.interpolate(x, scale_factor=up, mode="bilinear", align_corners=False)
    full = _empty((B, C, H, W), device=DEV)
    ops.bilinear_up_nchw(lg, full, up)
    interp_exact = bool(torch.equal(full.cpu(), x))
    pred = torch.argmax(x, dim=1)
    probs = F.softmax(x, dim=1).max(dim=1)[0]
    pred[probs < 0.5] = 127
    sig = torch.sigmoid(x)
    mism = int((pred != ids.cpu().long()).sum())
    cnt_ref = torch.stack([torch.bincount(pred[b].flatten(), minlength=C) for b in range(B)])
    over_ref = (sig >= 0.5).flatten(2).sum(-1)
    c = counts.cpu().long()
    info = {"name": f"logits_to_ids up={up}", "interp_bit_exact": interp_exact, "id_mismatch": mism,
            "count_mismatch": int((c[:, 0] != cnt_ref).sum()), "over_mismatch": int((c[:, 1] != over_ref).sum())}
    assert mism == 0 and info["count_mismatch"] == 0 and info["over_mismatch"] == 0, str(info)
    # merge filter
    cleaned = _empty_like(ids)
    ops.segment_filter(ids, counts, cleaned, count_th=512, overlap_th=0.5, ignore_label=127)
    cl_ref = pred.clone().numpy()
    pn, sg = pred.numpy(), sig.numpy()
    for b in range(B):
        cb = cl_ref[b]
        for lab, cnt in zip(*np.unique(pn[b], return_counts=True)):
            if cnt < 512 or lab in {-1, 127}:
                cb[cb == lab] = -1
                continue
            om = sg[b, lab] >= 0.5
            if (pn[b] == lab).sum() / om.sum() < 0.5:
                cb[cb == lab] = -1
    assert np.array_equal(cl_ref, cleaned.cpu().numpy()), "segment_filter mismatch"
    info["kept_labels"] = int(len(np.unique(cl_ref)) - 1)
    return info


def check_segment_filter_boundaries():
    """Merge filter (trainers_ldm_cond.py:1303-1325) at its decision boundaries, on constructed per-class counts:
    count == count_th is kept and count_th - 1 dropped (`count < count_th`), count / over == overlap_th exactly is kept
    and just below dropped (`< overlap_th`, float64 as numpy), over == 0 (numpy: x / 0 = inf) is kept, the ignore
    label and labels outside [0, C) are dropped."""
    C, count_th, overlap_th, ignore = 16, 100, 0.5, 15
    #            class: 0    1    2    3     4    5    6       7
    count = np.array([100,  99, 200, 200,  300, 500, 100,      0] + [0] * 7 + [400], np.int32)
    over = np.array([100, 100, 400, 401,    0, 100, 201,     50] + [0] * 7 + [400], np.int32)
    keep_ref = []
    for c in range(C):
        k = not (count[c] < count_th or c == ignore)
        if k and count[c] > 0:
            with np.errstate(divide="ignore"):
                if np.float64(count[c]) / np.float64(over[c]) < overlap_th:
                    k = False
        keep_ref.append(k and count[c] > 0)
    assert keep_ref[:8] == [True, False, True, False, True, True, False, False] and not keep_ref[15]
    ids = torch.from_numpy(np.concatenate([np.arange(-2, C + 2), np.arange(C)]).astype(np.int32)).view(1, -1).to(DEV)
    counts = torch.from_numpy(np.stack([count, over])[None]).contiguous().to(DEV)
    cleaned = _empty_like(ids)
    ops.segment_filter(ids, counts, cleaned, count_th=count_th, overlap_th=overlap_th, ignore_label=ignore)
    idn = ids.cpu().numpy()[0]
    want = np.array([i if (0 <= i < C and keep_ref[i]) else -1 for i in idn], np.int32)
    assert np.array_equal(cleaned.cpu().numpy()[0], want), (cleaned.cpu().numpy()[0].tolist(), want.tolist())
    return {"name": "segment_filter boundaries", "kept": int(sum(keep_ref))}


def check_bitmap():
    B, n, H, W = 2, 16, 24, 78
    rng = np.random.default_rng(0)
    ids_np = rng.integers(0, 60, size=(B, H, W)).astype(np.int32)
    ids_np[0, :2] = 31
    ids_np[1, 5:7] = 255
    ids = torch.from_numpy(ids_np).to(DEV)
    x = _empty((B, n, H, W), device=DEV)
    ops.encode_bitmap(ids, x, ignore_label=255, fill=0.5)
    t = torch.from_numpy(ids_np[0]).long()
    ign = t == 255
    ref = torch.remainder(torch.bitwise_right_shift(t, torch.arange(n)[:, None, None]), 2).float()
    ref[:, ign] = 0.5
    assert torch.equal(x[0].cpu(), ref), "encode_bitmap mismatch"
    dec = _empty((B, H, W), dtype=torch.int32, device=DEV)
    ops.decode_bitmap(x, dec, quirk31=True)
    exp = ids_np.copy()
    exp[exp == 31] = 0
    exp[ids_np == 255] = 65535
    assert np.array_equal(dec.cpu().numpy(), exp), "decode_bitmap mismatch"
    return {"name": "bitmap", "bit_exact": True}


def check_ccl():
    from scipy import ndimage
    B, H, W = 2, 96, 312
    rng = np.random.default_rng(1)
    sem = (rng.random((B, H, W)) < 0.55).astype(np.int32) * 13
    sem[1, 10:40, 20:200] = 13
    sem[1, 20:30, 50:150] = 2
    lab, nc = ops.ccl_label4(torch.from_numpy(sem).to(DEV), 13)
    lab, nc = lab.cpu().numpy(), nc.cpu().numpy()
    for b in range(B):
        ref, n = ndimage.label(sem[b] == 13)
        assert n == nc[b], f"ccl count {nc[b]} != {n}"
        assert np.array_equal(ref, lab[b]), "ccl labels differ from scipy.ndimage.label"
    return {"name": "ccl", "components": nc.tolist()}


def check_joint_hist():
    rng = np.random.default_rng(2)
    n = 384 * 1248
    a = (rng.integers(0, 19, n) * (1 << 20) + rng.integers(0, 30, n)).astype(np.int32)
    b = (rng.integers(0, 19, n) * (1 << 20) + rng.integers(0, 5, n)).astype(np.int32)
    a[:1000] = -1
    av, bv, c = ops.joint_hist(torch.from_numpy(a).to(DEV), torch.from_numpy(b).to(DEV), capacity=1 << 12)
    key = a.astype(np.int64) * (1 << 31) + b.astype(np.int64)
    uk, uc = np.unique(key, return_counts=True)
    got = av * (1 << 31) + bv
    assert np.array_equal(got, uk) and np.array_equal(c, uc), "joint_hist mismatch"
    # default (small) table: two overflow retries for these 54 150 pairs; and a frame-like case that fits at once
    av2, bv2, c2 = ops.joint_hist(torch.from_numpy(a).to(DEV), torch.from_numpy(b).to(DEV))
    assert np.array_equal(av2, av) and np.array_equal(bv2, bv) and np.array_equal(c2, c), "joint_hist retry mismatch"
    a3, b3 = (a // (1 << 20)).astype(np.int32), (b // (1 << 20)).astype(np.int32)
    av3, bv3, c3 = ops.joint_hist(torch.from_numpy(a3).to(DEV), torch.from_numpy(b3).to(DEV))
    uk3, uc3 = np.unique(a3.astype(np.int64) * (1 << 31) + b3.astype(np.int64), return_counts=True)
    assert np.array_equal(av3 * (1 << 31) + bv3, uk3) and np.array_equal(c3, uc3), "joint_hist (small table) mismatch"
    return {"name": "joint_hist", "pairs": int(len(uk))}


CHECKS = {
    "ddim": check_ddim,
    "layernorm_320": lambda: check_layernorm(320),
    "layernorm_1280": lambda: check_layernorm(1280, 468),
    # more row groups than resident warps (the persistent kernel's grid-stride loop + prefetch), ragged last group
    "layernorm_320_long": lambda: check_layernorm(320, 59905),
    "layernorm_640_long": lambda: check_layernorm(640, 14977),
    "layernorm_1280_long": lambda: check_layernorm(1280, 9001),
    "groupnorm_320": lambda: check_groupnorm(320),
    "groupnorm_960cat": lambda: check_groupnorm(640, 320, 1872),
    "groupnorm_1920cat_nosilu": lambda: check_groupnorm(1280, 640, 468, silu=False, eps=1e-6),
    # B = 8 at the 48x156 level: the cooperative two-sweep kernel; everything smaller: the one-pass cluster kernel
    "groupnorm_L0_b8_coop": lambda: check_groupnorm(320, 0, 7488, B=8),
    "groupnorm_L1_640_b8_tail": lambda: check_groupnorm(640, 0, 1872, B=8),   # slice longer than the register cache
    "groupnorm_L3_2560cat_b8": lambda: check_groupnorm(1280, 1280, 120, B=8),
    "groupnorm_L2_1280_b1": lambda: check_groupnorm(1280, 0, 468, B=1),       # 16 channel sets of two groups
    "groupnorm_L0_320_b1": lambda: check_groupnorm(320, 0, 7488, B=1),
    "groupnorm_ragged_hw": lambda: check_groupnorm(320, 0, 101, B=3),
    "groupnorm_tiny_hw": lambda: check_groupnorm(1280, 0, 5, B=2),            # fewer pixels than cluster ranks
    "groupnorm_cpg8": lambda: check_groupnorm(256, 0, 1000, B=1),
    "groupnorm_cpg4_cat": lambda: check_groupnorm(64, 64, 3000, B=2, silu=False),
    "gemv": check_gemv,
    "timestep_sinusoid": check_timestep_sinusoid,
    "conv_small_cin": check_conv_small_cin,
    "conv_out": check_conv_out,
    "gemm_conv_out_nchw": check_gemm_conv_out_nchw,
    "upsample_im2col": check_upsample_im2col,
    "vae_helpers": check_vae_helpers,
    "gemm_tiny": check_gemm_tiny,
    "gemm_plain_320": check_gemm_plain,
    "gemm_plain_f32_k1280": lambda: check_gemm_plain(777, 1280, 1280, f32out=True),
    "gemm_plain_bn256_multi_tile": lambda: check_gemm_plain(20000, 1280, 640, block_n=256),
    "gemm_plain_ktail": lambda: check_gemm_plain(300, 64, 72, residual=False),
    "gemm_conv3x3": check_gemm_conv3x3,
    "gemm_conv3x3_cat": lambda: check_gemm_conv3x3(2, 24, 78, 128, 64, 320),
    "gemm_conv3x3_L0": lambda: check_gemm_conv3x3(1, 48, 156, 320, 0, 320),
    "gemm_conv3x3_L3": lambda: check_gemm_conv3x3(3, 6, 20, 256, 0, 256),
    "gemm_concat_1x1": check_gemm_concat_1x1,
    "gemm_conv3x3_stride2": check_gemm_conv3x3_stride2,
    "gemm_conv3x3_stride2_odd": lambda: check_gemm_conv3x3_stride2(2, 12, 39, 256, 256),
    "gemm_conv3x3_stride2_L0": lambda: check_gemm_conv3x3_stride2(1, 48, 156, 320, 320),
    "gemm_conv3x3_stride2_pad0_silu": lambda: check_gemm_conv3x3_stride2(2, 32, 64, 128, 128, pad=0, silu=True),
    "gemm_conv3x3_stride2_pad0_odd": lambda: check_gemm_conv3x3_stride2(1, 13, 21, 64, 64, pad=0),
    "gemm_upsample_conv3x3": check_gemm_upsample_conv3x3,
    "gemm_upsample_conv3x3_L1": lambda: check_gemm_upsample_conv3x3(2, 24, 78, 640, 640),
    "gemm_upsample_conv3x3_L2_1280": lambda: check_gemm_upsample_conv3x3(1, 12, 39, 1280, 1280),
    "gemm_splitk_conv_L3_b1": check_gemm_splitk,
    "gemm_splitk_conv_L3_b8": lambda: check_gemm_splitk(8),
    "gemm_splitk_conv_L3_cat_b2": lambda: check_gemm_splitk(2, c1=1280, c2=1280, rowbias=False),
    "gemm_splitk_conv_L2_b1": lambda: check_gemm_splitk(1, 12, 39, 640, 0, 1280, residual=False),
    "gemm_splitk_1x1_k5120_b1": lambda: check_gemm_splitk(1, 6, 20, 5120, 0, 1280, taps=1, rowbias=False),
    "gemm_geglu": check_gemm_geglu,
    "gemm_qkv_40": check_gemm_qkv,
    "gemm_qkv_160": lambda: check_gemm_qkv(1, 8, 160, 468),
    # seq % 8 == 0: V^T leaves through the per-warp transpose (16-byte stores); image boundaries inside a warp's rows
    "gemm_qkv_40_vec": lambda: check_gemm_qkv(2, 8, 40, 304),
    "gemm_qkv_80_vec": lambda: check_gemm_qkv(3, 8, 80, 472),
    "gemm_qkv_40_vec_level0": lambda: check_gemm_qkv(1, 8, 40, 7488),
    "gemm_convt": check_gemm_convt,
    # LayerNorm folded into producer / consumer epilogues: QKV direct stores, QKV through TMA stores (whole 128-token
    # tiles of one image), 80- and 160-wide heads, GEGLU staged; a large row mean (cancellation in the mean term)
    "ln_fold_qkv_40": check_ln_fold,
    "ln_fold_qkv_40_level0": lambda: check_ln_fold("qkv", 1, 8, 40, 7488),
    "ln_fold_qkv_80": lambda: check_ln_fold("qkv", 2, 8, 80, 472),
    "ln_fold_qkv_160_big_mean": lambda: check_ln_fold("qkv", 2, 8, 160, 120, mean_shift=4.0),
    "ln_fold_geglu_320": lambda: check_ln_fold("geglu", 2, 8, 40, 300),
    "ln_fold_geglu_1280": lambda: check_ln_fold("geglu", 3, 8, 160, 120),
    "attn_40_tail": check_attention,
    "attn_40_long": lambda: check_attention(1, 2, 40, 1872),
    "attn_40_fold_tail": lambda: check_attention(1, 2, 40, 300, log2_units=True),
    "attn_40_fold_long": lambda: check_attention(1, 2, 40, 1872, log2_units=True),
    "attn_40_fold_tiny": lambda: check_attention(1, 1, 40, 40, log2_units=True),
    "attn_40_fold_spread": lambda: check_attention(1, 2, 40, 1000, log2_units=True, spread=4.0),
    "attn_40_spread": lambda: check_attention(1, 2, 40, 1000, spread=4.0),
    "attn_80_fold": lambda: check_attention(1, 2, 80, 468, log2_units=True),
    "attn_80": lambda: check_attention(1, 2, 80, 468),
    "attn_160": lambda: check_attention(2, 2, 160, 120),
    "attn_160_b": lambda: check_attention(1, 2, 160, 468),
    "cross_attn_40_kv77": check_cross_attention,
    "cross_attn_40_kv128_long": lambda: check_cross_attention(1, 8, 40, 7488, 128),
    "cross_attn_80_kv257": lambda: check_cross_attention(2, 8, 80, 468, 257, 1024),
    "cross_attn_160_kv16": lambda: check_cross_attention(2, 8, 160, 120, 16, 64),
    **{f"attn_{kind}_{d}_{'cross' if cross else 'self'}": (lambda f=f, d=d, cross=cross: f(d, cross))
       for kind, f in (("needles", check_attn_needles), ("const_v", check_attn_const_v), ("flat", check_attn_flat))
       for d in (40, 80, 160) for cross in (False, True)},
    "attn_bound_40_level0": lambda: check_attention_bound(40, 7488),
    "attn_bound_80": lambda: check_attention_bound(80, 1872),
    "attn_bound_160": lambda: check_attention_bound(160, 468),
    # mean 16-64x the spread: E[x^2] - mean^2 cancellation, in both GroupNorm kernels (each entry asserts which one ran),
    # concat inputs, SiLU on and off
    "groupnorm_cancel_L0_b8_coop": lambda: check_groupnorm_cancel(320, 0, 7488, 8, True, "gn_fused_kernel"),
    "groupnorm_cancel_L0_b8_coop_nosilu": lambda: check_groupnorm_cancel(320, 0, 7488, 8, False, "gn_fused_kernel"),
    "groupnorm_cancel_L1_b8_coop": lambda: check_groupnorm_cancel(640, 0, 1872, 8, True, "gn_fused_kernel"),
    "groupnorm_cancel_L0_b1_cluster": lambda: check_groupnorm_cancel(320, 0, 7488, 1, False, "gn_cluster_kernel"),
    "groupnorm_cancel_960cat_b2_cluster": lambda: check_groupnorm_cancel(640, 320, 1872, 2, True, "gn_cluster_kernel"),
    "groupnorm_cancel_L3_2560cat_b8_cluster_nosilu":
        lambda: check_groupnorm_cancel(1280, 1280, 120, 8, False, "gn_cluster_kernel"),
    "layernorm_cancel_320": lambda: check_layernorm_cancel(320, 20000),
    "layernorm_cancel_640": lambda: check_layernorm_cancel(640, 5000),
    "layernorm_cancel_1280": lambda: check_layernorm_cancel(1280, 2000),
    "logits_to_ids_up2": check_logits_to_ids,
    "logits_to_ids_up1": lambda: check_logits_to_ids(1),
    "segment_filter_boundaries": check_segment_filter_boundaries,
    "bitmap": check_bitmap,
    "ccl": check_ccl,
    "joint_hist": check_joint_hist,
}
