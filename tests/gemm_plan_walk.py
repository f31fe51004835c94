"""fp64 reference of the contraction kernel (ldm_gemm_bf16, ops.gemm) and a checked walk over the ops.gemm launches of
the production plans. Used by tests/test_gemm_plan_launches_gpu.py, tests/test_gemm_bound_controls.py (CPU) and
tools/gemm_launch_configs.py.

The reference is written from the contract in include/ldmseg_b200.h and the ops.gemm docstring. It calls nothing from
ops and reuses no kernel helper: it takes the bf16 / fp32 operands the kernel read (snapshots taken before the launch)
and computes in float64 on their device. Every mode the plans use is covered: plain and 1x1 with the a2 concat, 3x3
(stride 1 pad 1, stride 2 with a_pad 0 or 1) as nine shifted matmuls over a zero-padded copy of one image at a time,
up2 with the folded weights as given, bias / rowbias / residual, SiLU, GEGLU, the QKV split with part0, CONVT_LN_SILU,
row_stats and the LayerNorm fold, OUT_F32 and OUT_NCHW_F32 with n_store.

Two criteria, both against the reference:
  elementwise  |got - ref| <= r |ref| + a mag       (gpu_kernel_checks.bound_ratio, at BOUND_HEADROOM)
  per tile     rms(got - ref) <= KAPPA rms(bf16(ref) - ref) + floor     (bf16 outputs; 128 pixels x block_n columns)
mag is the same operation on absolute values. The elementwise bound grows with mag / |ref| ~ sqrt(K), so on long K it
cannot see one dropped K block; the tile criterion compares against the rounding noise of the tile instead.
"""
import math
from dataclasses import dataclass

import torch

import gpu_kernel_checks as GK

U = GK.U_BF16
bf16, f32, f64 = torch.bfloat16, torch.float32, torch.float64

# flag bits of ldm_gemm_flags (include/ldmseg_b200.h), restated so that the reference does not read them from the library
OUT_F32, GEGLU, QKV_SPLIT, SILU, CONVT_LN_SILU, OUT_NCHW_F32 = 1, 2, 4, 8, 16, 32
BLOCK_M = 128       # output pixels per tile (kBlockM)

# ---------------------------------------------------------------------------------------------------------- bounds
# fp32 accumulation. bf16 x bf16 products are exact in fp32. Nobody has measured whether the tcgen05 accumulator
# rounds to nearest on every add, so allow each of the K adds (and the epilogue's bias / rowbias / residual adds) an
# error of two ulps of the running sum, 2^-22 relative: one ulp for truncation instead of rounding, one for an internal
# alignment of partial sums inside an MMA. The running sum never exceeds mag, so |acc - exact| <= gamma(K) mag.
ACC_ULPS = 2.0 ** -22


def acc_gamma(K):
    return (K + 4) * ACC_ULPS


# SiLU in the kernel is h tanh(h) + h with h = x / 2 and tanh.approx.f32, whose relative error the PTX ISA gives as
# 2^-10.987: |error| <= 2^-10.9 |h tanh h| <= 2^-11.9 |x|.
SILU_APPROX = 2.0 ** -11.9
SILU_SLOPE = 1.1      # max |silu'(x)| = 1.0998
GELU_SLOPE = 1.13     # max |gelu'(x)| = 1.1289 (erf form)
# GELU in the kernel: Abramowitz-Stegun 7.1.26 erf (|abs err| < 1.5e-7) with ex2.approx (2^-22 rel) and rcp.approx:
# |gelu error| <= 2^-21 |g|, i.e. 2^-20 of |v| 1.13 mag_g with room to spare.
GELU_APPROX = 2.0 ** -20
# LayerNorm fold: mean and E[x^2] come from fp32 sums of 32-column partials (<= 32 + 40 sequential adds), relative
# error <= 72 * 2^-24 < 2^-17.8 of sum |x| and of sum x^2. var = E[x^2] - mean^2 then errs by 2^-17.8 E[x^2], rstd by
# half that relative to var: delta_rstd <= 2^-18.8 E[x^2] / var; the mean errs by 2^-17.8 mean|x| <= 2^-17.8 rms(x).
LN_STATS = 2.0 ** -17.8
# CONVT_LN_SILU: LayerNorm2d over cout <= 256 channels of the fp32 accumulator, two-pass in fp32: the mean and the
# variance err by <= cout 2^-24 relative (2^-16), rstd by half of it.
CONVT_STATS = 2.0 ** -16
# headroom of the elementwise criterion (gpu_kernel_checks.BOUND_HEADROOM = 1/4). Rounding the output errs by u |ref|
# + u |acc - ref|; everything before it by at most gamma mag + eps_epi. With mag >= |ref| (true for every mode here),
# (u |ref| + (1 + u)(gamma mag + e)) / (u |ref| + a mag') <= 1/4 when a mag' = 3u mag + 4.1 (gamma mag + e): the
# bf16 output rounding alone stays under a quarter of the bound and the pre-rounding error budget is used four times.
A_OUT_BF16 = 3 * U
A_OUT_F32 = 3 * 2.0 ** -24
# per-tile criterion: bf16(acc) is the bf16 value nearest acc, so |bf16(acc) - ref| <= |bf16(ref) - ref| + 2 |acc - ref|
# elementwise, and by Minkowski rms(got - ref) <= rms(bf16(ref) - ref) + 2 rms(acc - ref): kappa = 1 if the floor bounds
# rms(acc - ref). The floor uses a model of the accumulation error, not its worst case (that would be as loose as the
# elementwise bound): K adds, all of the same sign, of up to two ulps of a running sum whose size is that of a random
# walk, mag / sqrt(K), i.e. sqrt(K) 2^-22 rms(mag), plus the epilogue's approximation errors. Double rounding (exact ->
# fp32 -> bf16) and the model's slack take KAPPA to 1.25.
KAPPA = 1.25
TILE_FLOOR_ABS = 2.0 ** -30


@dataclass
class Out:
    """Reference of one output of a launch: ref / mag (fp64, the shape of the written region), the elementwise a and
    the per-element error terms of the tile floor."""
    ref: torch.Tensor
    mag: torch.Tensor
    a: float
    bf16_out: bool
    epi: torch.Tensor = None        # per-element approximation error bound of the epilogue (SiLU, GELU, LN stats)
    K: int = 0

    def mag_eff(self):
        """mag with the epilogue's absolute error terms folded in, for gpu_kernel_checks.bound_ratio (a mag_eff =
        a mag + 4.1 epi)."""
        return self.mag if self.epi is None else self.mag + 4.1 * self.epi / self.a


# ---------------------------------------------------------------------------------------------------------- contraction
def _mm(x, w):
    """x [rows, C] @ w[N, C]^T and |x| @ |w|^T in fp64."""
    xd, wd = x.to(f64), w.to(f64)
    return xd @ wd.t(), xd.abs() @ wd.abs().t()


def contraction(a1, w, a2=None, taps=1, a_stride=1, a_pad=1, up2=False, out_hw=None):
    """sum_{tap,c} A[b, y+dy, x+dx, c] W[n, tap (c1+c2) + c] in fp64 and the same on absolute values.
    a1 / a2: [B, H, W, C] (or [rows, C] for taps == 1); returns (acc, mag) of shape [B, Ho, Wo, N] ([rows, N] for 2-D
    inputs; up2: [B, 2H, 2W, N / 4]). out_hw: the output extents for a_stride = 2."""
    a = a1 if a2 is None else torch.cat([a1, a2], dim=-1)
    N = w.shape[0]
    if taps == 1:
        acc, mag = _mm(a.reshape(-1, a.shape[-1]), w)
        return acc.view(*a.shape[:-1], N), mag.view(*a.shape[:-1], N)
    B, H, W, C = a.shape
    if up2:
        cout = N // 4
        acc = torch.zeros((B, 2 * H, 2 * W, cout), dtype=f64, device=a.device)
        mag = torch.zeros_like(acc)
    else:
        Ho, Wo = (H, W) if a_stride == 1 else out_hw
        acc = torch.zeros((B, Ho, Wo, N), dtype=f64, device=a.device)
        mag = torch.zeros_like(acc)
    for b in range(B):   # one image at a time: the padded copy and the shifted views stay a few GB at most
        xp = torch.zeros((H + 3, W + 3, C), dtype=f64, device=a.device)
        if up2 or a_stride == 1 or a_pad == 1:
            xp[1:H + 1, 1:W + 1] = a[b].to(f64)      # zero padding 1 on every side (+ one spare row / column)
        else:
            xp[:H, :W] = a[b].to(f64)                # a_pad = 0: F.pad(x, (0, 1, 0, 1)), no padding in front
        xa = xp.abs()
        if up2:
            # class cls = 2 (row & 1) + (col & 1); tap (i, j) = 2i + j reads input (y + i - 1 + a, x + j - 1 + b)
            for cls in range(4):
                ca, cb = cls >> 1, cls & 1
                wc = w[cls * cout:(cls + 1) * cout].to(f64)
                s, m = 0.0, 0.0
                for i in range(2):
                    for j in range(2):
                        t = 2 * i + j
                        wt = wc[:, t * C:(t + 1) * C]
                        v = xp[i + ca:i + ca + H, j + cb:j + cb + W].reshape(-1, C)
                        va = xa[i + ca:i + ca + H, j + cb:j + cb + W].reshape(-1, C)
                        s = s + v @ wt.t()
                        m = m + va @ wt.abs().t()
                acc[b, ca::2, cb::2] = s.view(H, W, cout)
                mag[b, ca::2, cb::2] = m.view(H, W, cout)
            continue
        wd = w.to(f64)
        st = a_stride
        for ky in range(3):
            for kx in range(3):
                t = 3 * ky + kx
                wt = wd[:, t * C:(t + 1) * C]
                # stride 1 / a_pad 1: output (y, x) reads padded (st y + ky, st x + kx); a_pad 0: input (2y + ky, ...)
                v = xp[ky:ky + st * (Ho - 1) + 1:st, kx:kx + st * (Wo - 1) + 1:st].reshape(-1, C)
                va = xa[ky:ky + st * (Ho - 1) + 1:st, kx:kx + st * (Wo - 1) + 1:st].reshape(-1, C)
                acc[b] += (v @ wt.t()).view(Ho, Wo, N)
                mag[b] += (va @ wt.abs().t()).view(Ho, Wo, N)
    return acc, mag


def _silu(x):
    return x * torch.sigmoid(x)


def _gelu(x):
    return 0.5 * x * (1.0 + torch.erf(x / math.sqrt(2.0)))


def gemm_reference(c):
    """c: the snapshot of one ops.gemm call (see snapshot()). Returns {name: Out} for every output it writes:
    "out", or "q" / "k" / "vt" (the written regions [.., :d] / [:, :d, :seq]), and "row_stats" as (ref, bound) of the
    sums of the bf16 output the caller passes in later (row_stats_ref)."""
    flags, taps = c["flags"], c["taps"]
    a1, a2, w = c["a1"], c.get("a2"), c["w"]
    K = w.shape[1]
    gam = acc_gamma(K)
    out_hw = tuple(c["out"].shape[1:3]) if c.get("a_stride", 1) == 2 else None
    acc, mag = contraction(a1, w, a2, taps, c.get("a_stride", 1), c.get("a_pad", 1), c.get("up2", False), out_hw)
    res = {}
    if flags & CONVT_LN_SILU:
        B, H, W, _ = a1.shape
        N = w.shape[0]
        cout = N // 4
        g, be, eps = (t.to(f64) if torch.is_tensor(t) else t for t in c["ln"])
        v = acc + c["bias"].to(f64)                                   # [B, H, W, 4 cout], (dy, dx, co)
        v = v.view(B, H, W, 2, 2, cout)
        ma = mag.view(B, H, W, 2, 2, cout) + c["bias"].to(f64).abs().view(2, 2, cout)
        mean = v.mean(-1, keepdim=True)
        rstd = 1.0 / torch.sqrt((v - mean).pow(2).mean(-1, keepdim=True) + eps)
        xn = (v - mean) * rstd
        pre = g * xn + be
        ref = _silu(pre)
        # the LayerNorm of an accumulator that errs by gamma mag: xn errs by rstd gamma (mag + mean(mag)), and by
        # CONVT_STATS |xn| through the fp32 moments
        err_x = rstd * gam * (ma + ma.mean(-1, keepdim=True)) + CONVT_STATS * xn.abs()
        m = SILU_SLOPE * ((g * xn).abs() + be.abs() + g.abs() * err_x)
        epi = SILU_APPROX * pre.abs() + SILU_SLOPE * g.abs() * CONVT_STATS * xn.abs()
        perm = lambda t: t.permute(0, 1, 3, 2, 4, 5).reshape(B, 2 * H, 2 * W, cout)   # pixel shuffle
        res["out"] = Out(perm(ref), perm(m), A_OUT_BF16 + 4.1 * gam, True, perm(epi), K)
        return res
    pre = acc
    mpre = mag
    epi = None
    if c.get("ln_fold") is not None:
        # LN(x) W^T + b = rstd (x (gamma o W)^T - mean g) + b': x is a1 itself (the producer's bf16 rows)
        colsum, eps = c["ln_fold"][1].to(f64), c["ln_fold"][2]
        x = a1.reshape(-1, a1.shape[-1]).to(f64)
        mean = x.mean(-1, keepdim=True)
        ex2 = x.pow(2).mean(-1, keepdim=True)
        var = (ex2 - mean.pow(2)).clamp_min(0)
        rstd = 1.0 / torch.sqrt(var + eps)
        acc2 = acc.reshape(x.shape[0], -1)
        pre = rstd * (acc2 - mean * colsum)
        mpre = rstd * (mag.reshape(x.shape[0], -1) + mean.abs() * colsum.abs())
        # stats error: delta_rstd |rstd (acc - mean g)| + rstd |g| 2^-17.8 rms(x)
        epi = LN_STATS / 2 * (ex2 / (var + eps)) * pre.abs() + rstd * colsum.abs() * LN_STATS * ex2.sqrt()
        pre = pre.view(acc.shape)
        mpre = mpre.view(acc.shape)
        epi = epi.view(acc.shape)
    if c.get("bias") is not None:
        b = c["bias"].to(f64)
        if c.get("up2"):                 # [4 cout]: class cls's bias on the output pixels of parity class cls
            cout = b.numel() // 4
            pre, mpre = pre.clone(), mpre.clone()
            for cls in range(4):
                pre[:, cls >> 1::2, cls & 1::2] += b[cls * cout:(cls + 1) * cout]
                mpre[:, cls >> 1::2, cls & 1::2] += b[cls * cout:(cls + 1) * cout].abs()
        else:
            pre = pre + b
            mpre = mpre + b.abs()
    if c.get("rowbias") is not None:
        rb = c["rowbias"].to(f64)                       # [B, N]
        shp = [rb.shape[0]] + [1] * (pre.dim() - 2) + [rb.shape[1]]
        pre = pre + rb.view(shp)
        mpre = mpre + rb.abs().view(shp)
    if c.get("residual") is not None:
        r_ = c["residual"].to(f64).view(pre.shape)
        pre = pre + r_
        mpre = mpre + r_.abs()
    if flags & GEGLU:
        M = pre.numel() // pre.shape[-1]
        N = pre.shape[-1]
        p4 = pre.reshape(M, N // 32, 2, 16)
        m4 = mpre.reshape(M, N // 32, 2, 16)
        v, gt = p4[:, :, 0], p4[:, :, 1]
        mv, mg = m4[:, :, 0], m4[:, :, 1]
        gg = _gelu(gt)
        ref = (v * gg).reshape(M, N // 2)
        m = (mv * gg.abs() + v.abs() * GELU_SLOPE * mg).reshape(M, N // 2)
        e = (GELU_APPROX * v.abs() * GELU_SLOPE * mg).reshape(M, N // 2)
        if epi is not None:   # LN stats error of value and gate, through the product
            e4 = epi.reshape(M, N // 32, 2, 16)
            e = e + (e4[:, :, 0] * gg.abs() + v.abs() * GELU_SLOPE * e4[:, :, 1]).reshape(M, N // 2)
        res["out"] = Out(ref, m, A_OUT_BF16 + 4.1 * gam, True, e, K)
        return res
    if flags & SILU:
        e = SILU_APPROX * pre.abs() + (0 if epi is None else SILU_SLOPE * epi)
        pre, mpre, epi = _silu(pre), SILU_SLOPE * mpre, e
    if flags & QKV_SPLIT:
        q = c["qkv"]
        heads, d, seq = q["heads"], q["head_dim"], q["seq"]
        C = heads * d
        M = pre.numel() // pre.shape[-1]
        nparts = pre.shape[-1] // C
        nimg = M // seq
        pv = pre.reshape(nimg, seq, nparts, heads, d)
        mv = mpre.reshape(nimg, seq, nparts, heads, d)
        ev = None if epi is None else epi.reshape(nimg, seq, nparts, heads, d)
        for p in range(nparts):
            part = q.get("part0", 0) + p
            sel = lambda t: t[:, :, p].permute(0, 2, 1, 3).reshape(nimg * heads, seq, d)
            tr = (lambda t: t.transpose(1, 2)) if part == 2 else (lambda t: t)
            name = "qkv"[part] if part < 2 else "vt"
            res[name] = Out(tr(sel(pv)), tr(sel(mv)), A_OUT_BF16 + 4.1 * gam, True,
                            None if ev is None else tr(sel(ev)), K)
        return res
    if flags & OUT_NCHW_F32:
        ns = c["n_store"] or pre.shape[-1]
        t = lambda x: x[..., :ns].permute(0, 3, 1, 2)
        res["out"] = Out(t(pre), t(mpre), A_OUT_F32 + 4.1 * gam, False, None if epi is None else t(epi), K)
        return res
    if flags & OUT_F32:
        res["out"] = Out(pre, mpre, A_OUT_F32 + 4.1 * gam, False, epi, K)
        return res
    res["out"] = Out(pre, mpre, A_OUT_BF16 + 4.1 * gam, True, epi, K)
    return res


def row_stats_ref(out_bf16, rows):
    """row_stats of a bf16 [rows, N] output: per 32-column chunk and row, (sum, sum of squares) of the values as stored,
    part-major [ceil(N / 32), rows, 2], fp64; and the bound of the kernel's fp32 sums of 32 terms (32 2^-24 of the
    sums of absolute values)."""
    x = out_bf16.reshape(rows, -1).to(f64)
    N = x.shape[1]
    parts = (N + 31) // 32
    xp = torch.zeros((rows, parts * 32), dtype=f64, device=x.device)
    xp[:, :N] = x
    xs = xp.view(rows, parts, 32).transpose(0, 1)
    ref = torch.stack([xs.sum(-1), xs.pow(2).sum(-1)], -1)
    bound = 32 * 2.0 ** -24 * torch.stack([xs.abs().sum(-1), xs.pow(2).sum(-1)], -1) + 2.0 ** -60
    return ref, bound


# ---------------------------------------------------------------------------------------------------------- comparators
def _rows_cols(t, name):
    """[rows, cols] view of an output region for the tile criterion: rows = output pixels (tokens for q / k, channels x
    tokens transposed back for vt), cols = channels."""
    if name == "vt":
        t = t.transpose(-1, -2)
    return t.reshape(-1, t.shape[-1])


def elementwise_ratio(got, o):
    return GK.bound_ratio(got, o.ref, o.mag_eff(), U if o.bf16_out else 2.0 ** -24, o.a)


def tile_stats(got, o, name, block_n):
    """Per tile of 128 consecutive output rows x block_n columns: rms(got - ref) / (KAPPA rms(bf16(ref) - ref) +
    floor). Returns (worst ratio, its (row tile, column tile))."""
    g = _rows_cols(got.to(f64), name)
    r = _rows_cols(o.ref, name)
    m = _rows_cols(o.mag, name)
    e = None if o.epi is None else _rows_cols(o.epi, name)
    rows, cols = r.shape
    bn = max(1, min(block_n, cols))
    nt_r, nt_c = (rows + BLOCK_M - 1) // BLOCK_M, (cols + bn - 1) // bn
    pr, pc = nt_r * BLOCK_M - rows, nt_c * bn - cols

    def tile_ms(x):   # mean of squares per tile, and the count of elements
        x = torch.nn.functional.pad(x, (0, pc, 0, pr))
        return x.view(nt_r, BLOCK_M, nt_c, bn).pow(2).sum(dim=(1, 3))

    ones = torch.ones_like(r)
    n = tile_ms(ones)
    rms = lambda x: (tile_ms(x) / n).sqrt()
    err = rms(g - r)
    noise = rms(r.to(bf16).to(f64) - r)
    floor = 2 * math.sqrt(o.K) * ACC_ULPS * rms(m) + TILE_FLOOR_ABS * (1 + rms(m))
    if e is not None:
        floor = floor + 2 * rms(e)
    ratio = err / (KAPPA * noise + floor)
    ratio = torch.where(torch.isfinite(err), ratio, torch.full_like(ratio, float("inf")))
    worst = ratio.max().item()
    idx = divmod(int(ratio.argmax().item()), nt_c)
    return worst, idx


# ---------------------------------------------------------------------------------------------------------- snapshots
TENSOR_KEYS = ("a2", "bias", "rowbias", "residual")


def snapshot(a, k):
    """The operands of one ops.gemm(a1, w, out, **k) call, cloned before the launch (fp64 math happens later)."""
    a1, w = a[0], a[1]
    out = a[2] if len(a) > 2 else k.get("out")
    c = dict(a1=a1.clone(), w=w, out=out, flags=k.get("flags", 0), taps=k.get("taps", 1),
             a_stride=k.get("a_stride", 1), a_pad=k.get("a_pad", 1), up2=k.get("up2", False),
             n_store=k.get("n_store", 0), block_n=k.get("block_n", 0))
    for key in TENSOR_KEYS:
        v = k.get(key)
        c[key] = None if v is None else (v.clone() if key != "bias" else v)
    if k.get("ln") is not None:
        c["ln"] = k["ln"]
    if k.get("ln_fold") is not None:
        st, cs, eps = k["ln_fold"]
        c["ln_fold"] = (st.clone(), cs, eps)
    if k.get("qkv") is not None:
        c["qkv"] = dict(k["qkv"])
        c["qkv_before"] = {n: k["qkv"][n].clone() for n in ("q", "k", "vt") if k["qkv"].get(n) is not None}
    c["row_stats"] = k.get("row_stats")
    return c


def describe(a, k):
    """Descriptor summary of one ops.gemm(a1, w, out, **k) call (what tests/golden/gemm_launch_configs.json pins)."""
    a1, w = a[0], a[1]
    out = a[2] if len(a) > 2 else None
    rows = a1.numel() // a1.shape[-1]
    if k.get("a_stride", 1) == 2:
        rows = out.numel() // out.shape[-1]
    a2 = k.get("a2")
    d = dict(M=int(rows), N=int(w.shape[0]), K=int(w.shape[1]), taps=int(k.get("taps", 1)),
             c2=0 if a2 is None else int(a2.shape[-1]), flags=int(k.get("flags", 0)))
    if k.get("a_stride", 1) == 2:
        d["a_stride"], d["a_pad"] = 2, int(k.get("a_pad", 1))
    if k.get("up2"):
        d["up2"] = True
    for key in ("residual", "rowbias"):
        if k.get(key) is not None:
            d[key] = True
    if k.get("n_store"):
        d["n_store"] = int(k["n_store"])
    if k.get("block_n"):
        d["block_n_req"] = int(k["block_n"])
    q = k.get("qkv")
    if q is not None:
        d["qkv"] = dict(heads=q["heads"], d=q["head_dim"], seq=q["seq"], part0=q.get("part0", 0))
    if k.get("ln_fold") is not None:
        d["ln_fold"] = True
    if k.get("row_stats") is not None:
        d["row_stats"] = True
    return d


def qkv_straddles(desc):
    """True when some 128-row tile of a QKV launch holds tokens of two images (seq % 128 != 0 and more than one
    image): those tiles take the row-per-thread stores instead of the TMA path."""
    q = desc.get("qkv")
    return q is not None and q["seq"] % BLOCK_M != 0 and desc["M"] // q["seq"] > 1


# ---------------------------------------------------------------------------------------------------------- plans
EPILOGUES = {0: "staged", 1: "geglu", 2: "qkv", 3: "direct", 4: "convt", 5: "split", 6: "geglu_ln", 7: "qkv_ln"}
EPI_CODE = {"staged": "S", "geglu": "G", "qkv": "Q", "direct": "D", "convt": "C", "split": "K", "geglu_ln": "g",
            "qkv_ln": "q"}


def config_code(r):
    """One launch's selection as tests/golden/gemm_launch_configs.json pins it: epilogue letter (EPI_CODE), block_n,
    'p' for the CTA pair, '/split' for split-K. Example: K224p/3."""
    return f"{EPI_CODE.get(r['epilogue'], r['epilogue'])}{r['block_n']}{'p' if r['pair'] else ''}" + \
        (f"/{r['split']}" if r["split"] > 1 else "")
LATENT_HW = (48, 156)         # 384 x 1248 frames
MID_TIMESTEP = 481            # one mid-schedule DDIM timestep
# (plan, B, latent h, w, descriptor mode, ln_fold): the UNet plans the benchmark's configurations build (batch8 /
# clip8_strong / seq1101 run every B from 1 to 8 at 48x156, k2 runs B = 2 at 96x312), the LayerNorm-fold plan of
# bench.py --ln-fold, and the learnable-descriptor plan with its cross-attention context launches
UNET_PLANS = [(f"unet_remove_B{b}", b, 48, 156, "remove", False) for b in range(1, 9)] + [
    ("unet_remove_B2_96x312", 2, 96, 312, "remove", False),
    ("unet_lnfold_B8", 8, 48, 156, "remove", True),
    ("unet_learnable_B8", 8, 48, 156, "learnable", False),
]


def build_models(descriptors="remove", ln_fold=False, device="cuda"):
    """Models as tools/main_ldm.build_models / bench.py build them (same seeds), the UNet without its CUDA graph."""
    import copy
    from video_latent_diffusion_panoptic_segmentation_b200.tools import main_ldm
    p = copy.deepcopy(main_ldm.BASE)
    p["train_kwargs"]["image_descriptors"] = descriptors
    vae, unet, _ = main_ldm.build_models(p, torch.device(device), seed=0)
    unet.ln_fold = ln_fold
    unet.use_cuda_graph = False
    return p, vae, unet


def unet_plan(unet, B, h, w, device="cuda"):
    """The plan the sampler builds (split inputs x_t | rgb_latents, trainers_ldm_cond._loop_state) on seeded inputs at
    one mid-schedule timestep. Returns the plan state."""
    g = torch.Generator().manual_seed(1000 + B)
    parts = [torch.randn((B, 4, h, w), generator=g).to(device),
             (0.18215 * torch.randn((B, 4, h, w), generator=g)).to(device)]
    st = unet._get_plan(B, h, w, 8, parts=parts)
    st.timestep.fill_(MID_TIMESTEP)
    st.parts_keepalive = parts
    return st


def weight_names(*packed):
    """id(tensor) -> key of a packed weight (for launch names), over nested dicts / lists / tuples."""
    names = {}

    def visit(v, key):
        if torch.is_tensor(v):
            names.setdefault(id(v), key)
        elif isinstance(v, dict):
            for k2, v2 in v.items():
                visit(v2, f"{key}.{k2}" if key else str(k2))
        elif isinstance(v, list):
            for i, v2 in enumerate(v):
                visit(v2, f"{key}[{i}]")
        elif isinstance(v, tuple):
            for v2 in v:
                visit(v2, key)
    for p in packed:
        if p is not None:
            visit(p, "")
    return names


class Namer:
    """Readable, unique launch names: the packed weight's key (or, for a role-swapped GEMM, the key of its a1), a
    suffix for GEMMs of activations only, and #n for the n-th repetition of the same key."""

    def __init__(self, names):
        self.names, self.seen = names, {}

    def __call__(self, a, k):
        a1, w = a[0], a[1]
        key = self.names.get(id(w)) or (self.names.get(id(a1)) and self.names[id(a1)] + "^T") or "activations"
        if k.get("qkv") is not None:
            key += ".qkv" if k["qkv"].get("part0", 0) == 0 else ".kv"
        n = self.seen.get(key, 0)
        self.seen[key] = n + 1
        return key if n == 0 else f"{key}#{n}"


def kernel_names(fn):
    """(pair, epilogue) of every gemm_tc_kernel `fn` launches, in launch order (torch.profiler, CUDA activity)."""
    import re
    evs = [e for e in GK._kernel_events(fn) if "gemm_tc_kernel" in e.name]
    evs.sort(key=lambda e: getattr(getattr(e, "time_range", None), "start", 0))
    out = []
    for e in evs:
        m = re.search(r"gemm_tc_kernel<(true|false|1|0),\s*\(?(\d+)\)?>", e.name)
        out.append((m.group(1) in ("true", "1"), EPILOGUES.get(int(m.group(2)), m.group(2))) if m else (None, e.name))
    return out


def _run_gemm_plan(plan, on_gemm):
    from video_latent_diffusion_panoptic_segmentation_b200 import ops
    for fn, a, k in plan:
        if fn is ops.gemm:
            on_gemm(a, k)
        else:
            fn(*a, **k)


_MODELS, _PLANS = {}, {}


def plan_walks():
    """(plan name, builder) for every plan of UNET_PLANS, the seg-AE decoder and the RGB VAE encoder. builder(on_gemm) runs the plan once with every
    ops.gemm call routed through on_gemm(a, k, name) (which must launch it) and returns a dict with the final output
    ("out") and, for UNet plans, the model and plan state."""
    from video_latent_diffusion_panoptic_segmentation_b200 import ops
    real_gemm = ops.gemm

    def models(desc, fold):
        if (desc, fold) not in _MODELS:
            _MODELS.clear()
            _PLANS.clear()
            _MODELS[(desc, fold)] = build_models(desc, fold)
        return _MODELS[(desc, fold)]

    def unet_builder(B, h, w, desc, fold):
        def run(on_gemm):
            _, _, unet = models(desc, fold)
            if (B, h, w) not in _PLANS:     # one plan resident at a time
                _PLANS.clear()
                unet._plans.clear()
                _PLANS[(B, h, w)] = unet_plan(unet, B, h, w)
            st = _PLANS[(B, h, w)]
            namer = Namer(weight_names(unet._packed))
            route = lambda a, k: on_gemm(a, k, namer(a, k))
            _run_gemm_plan(st.ctx_plan, route)        # the context launches (learnable descriptors)
            _run_gemm_plan(st.plan, route)
            torch.cuda.synchronize()
            return {"out": st.out.clone(), "unet": unet, "st": st}
        return run

    def patched(fn, names):
        def run(on_gemm):
            namer = Namer(names())
            ops.gemm = lambda *a, **k: on_gemm(a, k, namer(a, k))
            try:
                out = fn()
            finally:
                ops.gemm = real_gemm
            torch.cuda.synchronize()
            return {"out": out}
        return run

    def segae():
        p, vae, _ = models("remove", False)
        g = torch.Generator().manual_seed(7)
        z = torch.randn((8, 4) + LATENT_HW, generator=g).cuda()

        def names():
            vae._pack() if vae._packed is None else None
            return weight_names(vae._packed)
        return patched(lambda: vae.decode_nhwc(z, scale=1.0 / vae.scaling_factor), names)

    def rgbvae():
        from video_latent_diffusion_panoptic_segmentation_b200.tools import main_ldm
        p, _, _ = models("remove", False)
        vim = main_ldm.build_vae_image(p, torch.device("cuda"), seed=0)
        g = torch.Generator().manual_seed(8)
        img = torch.rand((8, 3, 384, 1248), generator=g).cuda()

        def names():
            vim._pack() if vim._packed is None else None
            return weight_names(vim._packed)
        return patched(lambda: vim.encode_moments(img, scale=2.0, shift=-1.0), names)

    walks = [(n, unet_builder(B, h, w, desc, fold)) for n, B, h, w, desc, fold in UNET_PLANS]
    walks.append(("segae_decode_B8", lambda on_gemm: segae()(on_gemm)))
    walks.append(("rgbvae_encode_B8", lambda on_gemm: rgbvae()(on_gemm)))
    return walks


def config_walk(builder):
    """One run of a plan with every launch recorded: name, descriptor summary, (block_n, pair, split) and the
    (pair, epilogue) of the gemm_tc_kernel the profiler saw. No numerics."""
    from video_latent_diffusion_panoptic_segmentation_b200 import ops
    real_gemm = ops.gemm
    recs = []

    def on_gemm(a, k, name):
        real_gemm(*a, **k)
        bn, pair, split = ops.gemm_last_config()
        recs.append(dict(name=name, desc=describe(a, k), block_n=bn, pair=pair, split=split))

    builder(lambda a, k, name: real_gemm(*a, **k))       # build the plan (and warm up) outside the profiler
    for _ in range(3):   # a capture that lost a kernel record is taken again (the launches are deterministic)
        recs.clear()
        kn = kernel_names(lambda: builder(on_gemm))
        if len(kn) == len(recs):
            break
    assert len(kn) == len(recs), f"{len(kn)} gemm_tc_kernel launches seen for {len(recs)} ops.gemm calls"
    for r, (kpair, epi) in zip(recs, kn):
        assert kpair is None or kpair == r["pair"], f"{r['name']}: profiler saw pair={kpair}, last_config pair={r['pair']}"
        r["epilogue"] = epi
    return recs
