"""Torch-tensor front-ends of the C-ABI kernels. PyTorch here is plumbing only: device memory, streams.

Every function takes CUDA tensors, validates dtype/contiguity, and enqueues the kernel on the current stream.
Activations are NHWC bf16 (``[B, H, W, C]``); see include/ldmseg_b200.h for the per-op contracts.
"""
import ctypes as C

import torch

from . import _lib as L

bf16, f32, i32, i64 = torch.bfloat16, torch.float32, torch.int32, torch.int64


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _chk(t, dtype, name):
    if t is None:
        return
    if not t.is_cuda:
        raise L.LdmError(f"{name}: expected a CUDA tensor (no CPU fallback)")
    if t.dtype != dtype:
        raise L.LdmError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise L.LdmError(f"{name}: expected a contiguous tensor")


_EYE = {}


def _identity(device):
    """bf16 [256,256] identity shared by every GEMM on `device` (ldm_gemm_desc.identity)."""
    key = torch.device(device).index
    if key not in _EYE:
        _EYE[key] = torch.eye(256, dtype=bf16, device=device)
    return _EYE[key]


_SPLITK_WS = {}
SPLITK_WS_BYTES = 64 << 20   # fp32 partial tiles of the split-K launches


def _splitk_ws(device):
    """Split-K workspace shared by every GEMM on `device` (ldm_gemm_desc.splitk_ws). The launches that use it are
    ordered by the stream they run on: one stream at a time per device (the eager warm-up and the graph capture of a
    plan are sequential). Allocated at the first eager call, i.e. before any graph capture."""
    key = torch.device(device).index
    if key not in _SPLITK_WS:
        _SPLITK_WS[key] = torch.zeros(SPLITK_WS_BYTES, dtype=torch.uint8, device=device)
    return _SPLITK_WS[key]


def gemm(a1, w, out=None, *, a2=None, taps=1, bias=None, rowbias=None, residual=None, flags=0, block_n=0,
         qkv=None, ln=None, n_store=0, row_stats=None, ln_fold=None, a_stride=1, a_pad=1, up2=False):
    """out = epilogue(conv/gemm(a1 ++ a2, w)). a1/a2: [B,H,W,C] or [rows,C] bf16; w: [N, taps*(c1+c2)] bf16.

    qkv = dict(q=, k=, vt=, heads=, head_dim=, dpad=, seq=, seq_pad=[, part0=]) for LDM_GEMM_QKV_SPLIT (part0 and the
    number of C-wide column blocks of w select which of q / k / v are written: see ldm_gemm_desc.qkv_part0);
    ln = (gamma, beta, eps) for LDM_GEMM_CONVT_LN_SILU.
    LayerNorm fold (ldm_gemm_desc.ln_stats): row_stats = f32 [ceil(N/32), rows, 2] (part-major) written by the GEMM that produces x;
    ln_fold = (row_stats of x, colsum f32 [N], eps) on the QKV_SPLIT / GEGLU GEMM that consumes x with the folded
    weight / bias of fold_layernorm().
    a_stride = 2 (taps = 9): Conv2d(3x3, stride 2) of a1 [B, Hin, Win, C] into out [B, oh, ow, N] (a_pad = 1: padding 1;
    0: F.pad(0, 1, 0, 1) + padding 0), no im2col pass. up2 (taps = 4): nearest-upsample x2 + Conv2d(3x3, padding 1) of the
    low-resolution a1 into out [B, oh, ow, N / 4] with the class weights / bias of fold_upsample_conv3x3().
    """
    _chk(a1, bf16, "a1"); _chk(a2, bf16, "a2"); _chk(w, bf16, "w"); _chk(bias, f32, "bias")
    _chk(rowbias, f32, "rowbias"); _chk(residual, bf16, "residual")
    if a1.dim() == 2:
        B, H, W, c1 = 1, 1, a1.shape[0], a1.shape[1]
    else:
        B, H, W, c1 = a1.shape
    d = L.GemmDesc()
    d.a1, d.a2, d.w = _p(a1), _p(a2), _p(w)
    d.bias, d.rowbias, d.residual = _p(bias), _p(rowbias), _p(residual)
    if residual is not None:
        d.identity = _p(_identity(a1.device))
    ws = _splitk_ws(a1.device)
    d.splitk_ws, d.splitk_ws_bytes = _p(ws), ws.numel()
    if a_stride == 2:  # the GEMM's pixels are the OUTPUT pixels
        if out is None or out.dim() != 4 or a1.dim() != 4:
            raise L.LdmError("gemm: a_stride = 2 needs a1 [B, Hin, Win, C] and out [B, oh, ow, N]")
        d.a_stride, d.a_pad, d.a_H, d.a_W = 2, a_pad, H, W
        H, W = out.shape[1], out.shape[2]
    if up2:            # the GEMM's pixels are the INPUT pixels; out is the dense up-sampled tensor
        if out is None or out.dim() != 4 or a1.dim() != 4 or out.shape[-1] * 4 != w.shape[0]:
            raise L.LdmError("gemm: up2 needs a1 [B, H, W, C], out [B, oh, ow, cout] and w [4 * cout, 4 * C]")
        d.up2, d.out_H, d.out_W = 1, out.shape[1], out.shape[2]
    d.B, d.H, d.W, d.c1 = B, H, W, c1
    d.c2 = 0 if a2 is None else a2.shape[-1]
    d.N = w.shape[0]
    d.taps, d.block_n, d.flags = taps, block_n, flags
    if w.shape[1] != taps * (d.c1 + d.c2):
        raise L.LdmError(f"gemm: weight K={w.shape[1]} != taps*(c1+c2)={taps * (d.c1 + d.c2)}")
    if flags & L.LDM_GEMM_QKV_SPLIT:
        for k_ in ("q", "k", "vt"):
            _chk(qkv.get(k_), bf16, k_)
        d.q, d.k, d.vt = _p(qkv.get("q")), _p(qkv.get("k")), _p(qkv.get("vt"))
        d.heads, d.head_dim, d.dpad = qkv["heads"], qkv["head_dim"], qkv["dpad"]
        d.seq, d.seq_pad = qkv["seq"], qkv["seq_pad"]
        d.vt_rows = qkv["vt"].shape[1] if qkv.get("vt") is not None else 0
        d.qkv_part0 = qkv.get("part0", 0)
    else:
        _chk(out, f32 if flags & (L.LDM_GEMM_OUT_F32 | L.LDM_GEMM_OUT_NCHW_F32) else bf16, "out")
        d.out = _p(out)
        d.n_store = n_store
    if flags & L.LDM_GEMM_CONVT_LN_SILU:
        g, b_, eps = ln
        _chk(g, f32, "ln_gamma"); _chk(b_, f32, "ln_beta")
        d.ln_gamma, d.ln_beta, d.ln_eps = _p(g), _p(b_), eps
    if row_stats is not None:
        _chk(row_stats, f32, "row_stats")
        if row_stats.numel() != B * H * W * ((d.N + 31) // 32) * 2:
            raise L.LdmError(f"gemm: row_stats has {row_stats.numel()} floats, expected ceil(N/32) * rows * 2")
        d.row_stats_out = _p(row_stats)
    if ln_fold is not None:
        st, colsum, eps = ln_fold
        _chk(st, f32, "ln_stats"); _chk(colsum, f32, "ln_colsum")
        d.ln_parts = (c1 + 31) // 32
        if st.numel() != B * H * W * d.ln_parts * 2 or colsum.numel() != d.N:
            raise L.LdmError("gemm: ln_fold stats / colsum shape mismatch")
        d.ln_stats, d.ln_colsum, d.ln_fold_eps = _p(st), _p(colsum), eps
    L.check(L.lib().ldm_gemm_bf16(C.byref(d), _stream()), "ldm_gemm_bf16")
    return out


def fold_layernorm(w, bias, gamma, beta):
    """Weights of a Linear that follows a LayerNorm, for the folded form (ldm_gemm_desc.ln_stats). w: [N, C] in the
    layout the GEMM consumes (bf16 or f32; already packed / interleaved / scaled), bias: f32 [N] or None, gamma / beta:
    f32 [C]. Returns (w' bf16 [N, C] = gamma o w, bias' f32 [N] = bias + w beta, colsum f32 [N] = sum_c w'[n, c] of the
    ROUNDED w', so that the mean term cancels exactly against what the tensor core multiplies)."""
    wf = w.float()
    w2 = (wf * gamma.float()[None, :]).to(bf16)
    b2 = wf @ beta.float()
    if bias is not None:
        b2 = b2 + bias.float()
    return w2.contiguous(), b2.contiguous(), w2.float().sum(dim=1).contiguous()


def fold_upsample_conv3x3(w, bias):
    """Weights of Conv2d(3x3, padding 1) behind F.interpolate(scale 2, nearest), for ldm_gemm_desc.up2. w: [N, 3, 3, C]
    (or the packed [N, 9 * C], tap-major), bias f32 [N]. Output pixel (2y + a, 2x + b) only ever sees the input rows
    {y - 1 + a, y + a} and columns {x - 1 + b, x + b}: its nine taps collapse onto a 2x2 kernel whose entries are sums of
    the original ones (rows: a = 0 -> {k0, k1 + k2}, a = 1 -> {k0 + k1, k2}; columns likewise), summed in fp32 and rounded
    to bf16 once. Returns (w' bf16 [4 * N, 4 * C], class-major rows, taps (i, j) = 2 i + j; bias' f32 [4 * N])."""
    N = w.shape[0]
    w = w.float().reshape(N, 3, 3, -1)
    groups = {0: ([0], [1, 2]), 1: ([0, 1], [2])}
    out = []
    for a in (0, 1):
        for b in (0, 1):
            taps = []
            for i in (0, 1):
                for j in (0, 1):
                    taps.append(sum(w[:, ky, kx] for ky in groups[a][i] for kx in groups[b][j]))
            out.append(torch.stack(taps, dim=1).reshape(N, -1))
    return torch.cat(out, 0).to(bf16).contiguous(), bias.float().repeat(4).contiguous()


def gemm_last_config():
    """(block_n, pair, split_k) of this thread's last gemm launch."""
    bn, pr, sk = C.c_int32(), C.c_int32(), C.c_int32()
    L.lib().ldm_gemm_last_config(C.byref(bn), C.byref(pr), C.byref(sk))
    return bn.value, bool(pr.value), sk.value


def alloc_qkv(B, heads, seq, d, device):
    """Zero-padded head-split buffers for LDM_GEMM_QKV_SPLIT / flash_attn (see include/ldmseg_b200.h): q, k
    [B*heads, seq, dpad]; vt [B*heads, vt_rows, seq_pad] with the ones row at index d when d % 16 != 0."""
    dpad, seq_pad = (d + 63) // 64 * 64, (seq + 7) // 8 * 8
    rows = (d + 15) // 16 * 16
    q = torch.zeros((B * heads, seq, dpad), dtype=bf16, device=device)
    k = torch.zeros((B * heads, seq, dpad), dtype=bf16, device=device)
    vt = torch.zeros((B * heads, rows, seq_pad), dtype=bf16, device=device)
    if rows != d:
        vt[:, d, :seq] = 1.0
    return dict(q=q, k=k, vt=vt, heads=heads, head_dim=d, dpad=dpad, seq=seq, seq_pad=seq_pad)


def alloc_kv(B, heads, kv_seq, d, device):
    """Head-split key / value buffers of a cross-attention context of kv_seq tokens (LDM_GEMM_QKV_SPLIT with part0 = 1
    writes them; flash_attn(kv_seq=) reads them): k [B*heads, kv_seq, dpad], vt [B*heads, vt_rows, seq_pad]."""
    dpad, seq_pad = (d + 63) // 64 * 64, (kv_seq + 7) // 8 * 8
    rows = (d + 15) // 16 * 16
    k = torch.zeros((B * heads, kv_seq, dpad), dtype=bf16, device=device)
    vt = torch.zeros((B * heads, rows, seq_pad), dtype=bf16, device=device)
    if rows != d:
        vt[:, d, :kv_seq] = 1.0
    return dict(k=k, vt=vt, heads=heads, head_dim=d, dpad=dpad, seq=kv_seq, seq_pad=seq_pad)


def flash_attn(q, k, vt, out, *, B, heads, seq, head_dim, dpad, seq_pad, scale, kv_seq=0):
    """kv_seq > 0: cross-attention, k [B*heads, kv_seq, dpad], vt [B*heads, vt_rows, seq_pad >= kv_seq]."""
    for t, n in ((q, "q"), (k, "k"), (vt, "vt"), (out, "out")):
        _chk(t, bf16, n)
    d = L.AttnDesc()
    d.q, d.k, d.vt, d.out = _p(q), _p(k), _p(vt), _p(out)
    d.B, d.heads, d.seq, d.head_dim, d.dpad, d.seq_pad, d.scale = B, heads, seq, head_dim, dpad, seq_pad, scale
    d.kv_seq = kv_seq
    d.vt_rows = vt.shape[1]
    L.check(L.lib().ldm_flash_attn_fwd(C.byref(d), _stream()), "ldm_flash_attn_fwd")
    return out


def groupnorm(x1, gamma, beta, out, stats, *, x2=None, groups=32, eps=1e-5, silu=True):
    _chk(x1, bf16, "x1"); _chk(x2, bf16, "x2"); _chk(gamma, f32, "gamma"); _chk(beta, f32, "beta")
    _chk(out, bf16, "out"); _chk(stats, f32, "stats")
    B = x1.shape[0]
    c1 = x1.shape[-1]
    HW = x1.numel() // (B * c1)
    d = L.GroupNormDesc()
    d.x1, d.x2, d.gamma, d.beta, d.out, d.stats = _p(x1), _p(x2), _p(gamma), _p(beta), _p(out), _p(stats)
    d.B, d.HW, d.c1, d.c2 = B, HW, c1, (0 if x2 is None else x2.shape[-1])
    d.groups, d.eps, d.silu = groups, eps, int(silu)
    if stats.numel() * 4 < L.lib().ldm_groupnorm_scratch_bytes(B, groups):
        raise L.LdmError("groupnorm: stats scratch too small (see gn_scratch)")
    L.check(L.lib().ldm_groupnorm_silu(C.byref(d), _stream()), "ldm_groupnorm_silu")
    return out


def gn_scratch(B, groups, device):
    # zeros: the tail of the scratch holds the fused kernel's barrier counters (zero before first use, left zero)
    return torch.zeros(L.lib().ldm_groupnorm_scratch_bytes(B, groups) // 4, dtype=f32, device=device)


def layernorm(x, gamma, beta, out, eps=1e-5):
    _chk(x, bf16, "x"); _chk(gamma, f32, "gamma"); _chk(beta, f32, "beta"); _chk(out, bf16, "out")
    Cc = x.shape[-1]
    L.check(L.lib().ldm_layernorm(_p(x), _p(gamma), _p(beta), _p(out), x.numel() // Cc, Cc, eps, _stream()),
            "ldm_layernorm")
    return out


def timestep_sinusoid(timesteps, t_index, freqs, out):
    _chk(timesteps, i64, "timesteps"); _chk(t_index, i32, "t_index"); _chk(freqs, f32, "freqs"); _chk(out, f32, "out")
    L.check(L.lib().ldm_timestep_sinusoid(_p(timesteps), _p(t_index), _p(freqs), _p(out), freqs.numel(), _stream()),
            "ldm_timestep_sinusoid")
    return out


def gemv(w, x, out, bias=None, bias2=None, silu=False):
    _chk(w, bf16, "w"); _chk(x, f32, "x"); _chk(out, f32, "out"); _chk(bias, f32, "bias"); _chk(bias2, f32, "bias2")
    L.check(L.lib().ldm_gemv_bf16(_p(w), _p(bias), _p(bias2), _p(x), _p(out), w.shape[0], w.shape[1], int(silu),
                                  _stream()), "ldm_gemv_bf16")
    return out


def timestep_sinusoid_rows(timesteps, freqs, out):
    """timesteps int64 [B] -> out f32 [B, 2 * half]; row b equals timestep_sinusoid of timesteps[b] bit for bit."""
    _chk(timesteps, i64, "timesteps"); _chk(freqs, f32, "freqs"); _chk(out, f32, "out")
    B = timesteps.numel()
    if out.numel() != B * 2 * freqs.numel():
        raise L.LdmError(f"timestep_sinusoid_rows: out has {out.numel()} elements, expected {B} x {2 * freqs.numel()}")
    L.check(L.lib().ldm_timestep_sinusoid_rows(_p(timesteps), _p(freqs), _p(out), freqs.numel(), B, _stream()),
            "ldm_timestep_sinusoid_rows")
    return out


def gemv_rows(w, x, out, bias=None, bias2=None, silu=False, seg_offs=None):
    """x f32 [B, K] -> out f32: row b equals gemv of x[b] bit for bit. out is [B, N], or with seg_offs (device int32
    [nseg + 1], ascending column offsets from 0 to N) segment-major: segment s is a contiguous [B, width_s] block at
    offset seg_offs[s] * B (ldm_gemv_bf16_rows)."""
    _chk(w, bf16, "w"); _chk(x, f32, "x"); _chk(out, f32, "out"); _chk(bias, f32, "bias"); _chk(bias2, f32, "bias2")
    _chk(seg_offs, i32, "seg_offs")
    N, K = w.shape
    B = x.numel() // K
    if x.numel() != B * K or out.numel() != B * N:
        raise L.LdmError(f"gemv_rows: x has {x.numel()} and out {out.numel()} elements for w [{N}, {K}]")
    nseg = 0 if seg_offs is None else seg_offs.numel() - 1
    L.check(L.lib().ldm_gemv_bf16_rows(_p(w), _p(bias), _p(bias2), _p(x), _p(out), N, K, B, _p(seg_offs), nseg,
                                       int(silu), _stream()), "ldm_gemv_bf16_rows")
    return out


def _check_rows(what, sample, rows, elems_per_image, named):
    """Shared checks of the *_step_rows wrappers: dtypes, element counts, one int32 row per (possibly partial) image."""
    for t, nm in named:
        _chk(t, f32, nm)
    _chk(sample, f32, "sample"); _chk(rows, i32, "rows")
    n = sample.numel()
    for t, nm in named:
        if nm != "coef" and t is not None and t.numel() != n:
            raise L.LdmError(f"{what}: {nm} has {t.numel()} elements, sample {n}")
    if elems_per_image <= 0 or elems_per_image % 4 or rows.numel() < -(-n // elems_per_image):
        raise L.LdmError(f"{what}: elems_per_image={elems_per_image} (a positive multiple of 4) and one row per image "
                         f"({rows.numel()} rows for {n} elements)")
    return n


def ddim_step_rows(eps, sample, coef, rows, elems_per_image, prev_sample=None, pred_x0=None):
    """ddim_step without guidance or clipping, element i at coefficient row rows[i // elems_per_image] (the timestep
    value, as t_index)."""
    n = _check_rows("ddim_step_rows", sample, rows, elems_per_image,
                    ((eps, "eps"), (coef, "coef"), (prev_sample, "prev"), (pred_x0, "x0")))
    L.check(L.lib().ldm_ddim_step_rows(_p(eps), _p(sample), _p(coef), _p(rows), _p(prev_sample), _p(pred_x0), n,
                                       elems_per_image, _stream()), "ldm_ddim_step_rows")


def dpmpp_step_rows(eps, sample, coef, rows, elems_per_image, prev_sample, x0_prev):
    """dpmpp_step without guidance, element i at row rows[i // elems_per_image] of coef (the step index)."""
    n = _check_rows("dpmpp_step_rows", sample, rows, elems_per_image,
                    ((eps, "eps"), (coef, "coef"), (prev_sample, "prev"), (x0_prev, "x0_prev")))
    if coef.dim() != 2 or coef.shape[1] != 8:
        raise L.LdmError("dpmpp_step_rows: coef must be [steps, 8]")
    L.check(L.lib().ldm_dpmpp_step_rows(_p(eps), _p(sample), _p(coef), _p(rows), _p(prev_sample), _p(x0_prev), n,
                                        elems_per_image, _stream()), "ldm_dpmpp_step_rows")


def unipc_step_rows(eps, sample, coef, rows, elems_per_image, prev_sample, last, history):
    """unipc_step without guidance, element i at row rows[i // elems_per_image] of coef (the step index)."""
    history = list(history)
    order = len(history)
    if not 1 <= order <= 3:
        raise L.LdmError(f"unipc_step_rows: history holds the x0 predictions of solver orders 1 to 3, got {order}")
    n = _check_rows("unipc_step_rows", sample, rows, elems_per_image,
                    ((eps, "eps"), (coef, "coef"), (prev_sample, "prev"), (last, "last"),
                     *((m, f"m{k + 1}") for k, m in enumerate(history))))
    owned = [last] + history
    if len({t.data_ptr() for t in owned}) != len(owned) or any(
            t.data_ptr() in (sample.data_ptr(), prev_sample.data_ptr()) for t in owned):
        raise L.LdmError("unipc_step_rows: last and the history buffers must not alias each other, sample or prev")
    if coef.dim() != 2 or coef.shape[1] != 20:
        raise L.LdmError("unipc_step_rows: coef must be [steps, 20]")
    m = history + [None] * (3 - order)
    L.check(L.lib().ldm_unipc_step_rows(_p(eps), _p(sample), _p(coef), _p(rows), _p(prev_sample), _p(last), _p(m[0]),
                                        _p(m[1]), _p(m[2]), order, n, elems_per_image, _stream()),
            "ldm_unipc_step_rows")


def pack_small_cin_weight(w):
    """Conv2d weight [cout, cin, 3, 3] (reference layout) -> f32 [cin, 3, 3, cout] for conv3x3_small_cin."""
    return w.detach().to(f32).permute(1, 2, 3, 0).contiguous()


def conv3x3_small_cin(srcs, w, bias, out, scale=1.0, silu=False, shift=0.0):
    """srcs: list of 1..3 f32 NCHW [B,cps,h,w], mapped to x*scale + shift on the fly; w f32 [len(srcs)*cps, 3, 3, cout]
    (pack_small_cin_weight); out bf16 NHWC [B,h,w,cout]; silu: SiLU on the result."""
    for s in srcs:
        _chk(s, f32, "src")
    _chk(w, f32, "w"); _chk(bias, f32, "bias"); _chk(out, bf16, "out")
    B, cps, h, wd = srcs[0].shape
    s = list(srcs) + [None] * (3 - len(srcs))
    L.check(L.lib().ldm_conv3x3_small_cin_affine(_p(s[0]), _p(s[1]), _p(s[2]), len(srcs), cps, scale, shift, _p(w),
                                                 _p(bias), _p(out), B, h, wd, w.shape[-1], int(silu), _stream()),
            "ldm_conv3x3_small_cin_affine")
    return out


def conv_out(x, w, bias, out):
    """x bf16 NHWC [B,h,w,cin]; w f32 [cout,cin,3,3]; out f32 NCHW [B,cout,h,w]."""
    _chk(x, bf16, "x"); _chk(w, f32, "w"); _chk(bias, f32, "bias"); _chk(out, f32, "out")
    B, h, wd, cin = x.shape
    L.check(L.lib().ldm_conv_out(_p(x), _p(w), _p(bias), _p(out), B, h, wd, cin, w.shape[0], _stream()), "ldm_conv_out")
    return out


def ddim_step(eps, sample, coef, t_index, prev_sample=None, pred_x0=None, eps_text=None, guidance_scale=0.0,
              clip_sample_range=0.0, use_clipped_model_output=False):
    """eps_text given: eps <- eps + guidance_scale * (eps_text - eps) first (classifier-free guidance).
    clip_sample_range > 0: x0 clamped to +-range; use_clipped_model_output: eps re-derived from the clamped x0."""
    for t, n in ((eps, "eps"), (sample, "sample"), (coef, "coef"), (prev_sample, "prev"), (pred_x0, "x0"),
                 (eps_text, "eps_text")):
        _chk(t, f32, n)
    _chk(t_index, i32, "t_index")
    L.check(L.lib().ldm_ddim_step_clip(_p(eps), _p(eps_text), float(guidance_scale), _p(sample), _p(coef), _p(t_index),
                                       _p(prev_sample), _p(pred_x0), sample.numel(), float(clip_sample_range),
                                       int(bool(use_clipped_model_output)), _stream()), "ldm_ddim_step_clip")


def dpmpp_step(eps, sample, coef, step_index, prev_sample, x0_prev, eps_text=None, guidance_scale=0.0):
    """DPM-Solver++ update with the scalars of row *step_index of coef (f32 [steps, 8], DPMSolverMultistepScheduler):
    prev_sample <- solver step of sample, x0_prev <- this step's x0 (read first on second-order rows). eps_text given:
    classifier-free guidance first, as ddim_step. prev_sample may be sample."""
    for t, n in ((eps, "eps"), (sample, "sample"), (coef, "coef"), (prev_sample, "prev"), (x0_prev, "x0_prev"),
                 (eps_text, "eps_text")):
        _chk(t, f32, n)
    _chk(step_index, i32, "step_index")
    n = sample.numel()
    for t, name in ((eps, "eps"), (prev_sample, "prev"), (x0_prev, "x0_prev"), (eps_text, "eps_text")):
        if t is not None and t.numel() != n:
            raise L.LdmError(f"dpmpp_step: {name} has {t.numel()} elements, sample {n}")
    if coef.dim() != 2 or coef.shape[1] != 8 or step_index.numel() != 1:
        raise L.LdmError("dpmpp_step: coef must be [steps, 8] and step_index one int32 element")
    L.check(L.lib().ldm_dpmpp_step(_p(eps), _p(eps_text), float(guidance_scale), _p(sample), _p(coef), _p(step_index),
                                   _p(prev_sample), _p(x0_prev), n, _stream()), "ldm_dpmpp_step")


def unipc_step(eps, sample, coef, step_index, prev_sample, last, history, eps_text=None, guidance_scale=0.0):
    """UniPC update with the scalars of row *step_index of coef (f32 [steps, 20], UniPCMultistepScheduler): corrects
    the previous step's result with `last` (the sample that step started from, corrected), then predicts prev_sample.
    history = [m1, .., m_order], the previous x0 predictions, newest first; last and history are updated in place.
    eps_text given: classifier-free guidance first, as ddim_step. prev_sample may be sample."""
    history = list(history)
    order = len(history)
    if not 1 <= order <= 3:
        raise L.LdmError(f"unipc_step: history holds the x0 predictions of solver orders 1 to 3, got {order}")
    for t, nm in ((eps, "eps"), (sample, "sample"), (coef, "coef"), (prev_sample, "prev"), (last, "last"),
                  (eps_text, "eps_text"), *((m, f"m{k + 1}") for k, m in enumerate(history))):
        _chk(t, f32, nm)
    _chk(step_index, i32, "step_index")
    n = sample.numel()
    for t, name in ((eps, "eps"), (prev_sample, "prev"), (last, "last"), (eps_text, "eps_text"),
                    *((m, f"m{k + 1}") for k, m in enumerate(history))):
        if t is not None and t.numel() != n:
            raise L.LdmError(f"unipc_step: {name} has {t.numel()} elements, sample {n}")
    owned = [last] + history
    if len({t.data_ptr() for t in owned}) != len(owned) or any(
            t.data_ptr() in (sample.data_ptr(), prev_sample.data_ptr()) for t in owned):
        raise L.LdmError("unipc_step: last and the history buffers must not alias each other, sample or prev")
    if coef.dim() != 2 or coef.shape[1] != 20 or step_index.numel() != 1:
        raise L.LdmError("unipc_step: coef must be [steps, 20] and step_index one int32 element")
    m = history + [None] * (3 - order)
    L.check(L.lib().ldm_unipc_step(_p(eps), _p(eps_text), float(guidance_scale), _p(sample), _p(coef), _p(step_index),
                                   _p(prev_sample), _p(last), _p(m[0]), _p(m[1]), _p(m[2]), order, n, _stream()),
            "ldm_unipc_step")


def upsample_nearest(x, out):
    _chk(x, bf16, "x"); _chk(out, bf16, "out")
    B, h, w, Cc = x.shape
    L.check(L.lib().ldm_upsample_nearest(_p(x), _p(out), B, h, w, Cc, out.shape[1], out.shape[2], _stream()),
            "ldm_upsample_nearest")
    return out


def im2col3x3_s2(x, out, pad_lo=1):
    """pad_lo = 1: Conv2d(stride 2, padding 1); pad_lo = 0: F.pad(x, (0, 1, 0, 1)) + Conv2d(stride 2, padding 0)."""
    _chk(x, bf16, "x"); _chk(out, bf16, "out")
    B, h, w, Cc = x.shape
    oh, ow = (h + pad_lo - 2) // 2 + 1, (w + pad_lo - 2) // 2 + 1
    L.check(L.lib().ldm_im2col3x3_s2_pad(_p(x), _p(out), B, h, w, Cc, oh, ow, pad_lo, _stream()),
            "ldm_im2col3x3_s2_pad")
    return out


def softmax_rows(s, p, scale, cols=None):
    """p[r, :cols] = softmax(scale * s[r, :cols]); s f32 [rows, ld_s], p bf16 [rows, ld_p]."""
    _chk(s, f32, "s"); _chk(p, bf16, "p")
    cols = s.shape[1] if cols is None else cols
    L.check(L.lib().ldm_softmax_rows(_p(s), _p(p), s.shape[0], cols, s.shape[1], p.shape[1], scale, _stream()),
            "ldm_softmax_rows")
    return p


def resize_bilinear_planar(x, out):
    """x f32 [..., h, w] -> out f32 [..., oh, ow], F.interpolate(mode="bilinear", align_corners=False) per plane."""
    _chk(x, f32, "x"); _chk(out, f32, "out")
    h, w = x.shape[-2:]
    oh, ow = out.shape[-2:]
    L.check(L.lib().ldm_resize_bilinear_planar(_p(x), _p(out), x.numel() // (h * w), h, w, oh, ow, _stream()),
            "ldm_resize_bilinear_planar")
    return out


def logits_to_ids(logits, ids, counts, *, up, mask_th, ignore_label):
    """logits f32 NHWC [B,h,w,C]; ids i32 [B,up*h,up*w]; counts i32 [B,2,C]."""
    _chk(logits, f32, "logits"); _chk(ids, i32, "ids"); _chk(counts, i32, "counts")
    B, h, w, Cc = logits.shape
    L.check(L.lib().ldm_logits_to_ids(_p(logits), _p(ids), _p(counts), B, h, w, Cc, up, mask_th, ignore_label,
                                      _stream()), "ldm_logits_to_ids")
    return ids, counts


def bilinear_up_nchw(logits, out, up):
    _chk(logits, f32, "logits"); _chk(out, f32, "out")
    B, h, w, Cc = logits.shape
    L.check(L.lib().ldm_bilinear_up_nchw(_p(logits), _p(out), B, h, w, Cc, up, _stream()), "ldm_bilinear_up_nchw")
    return out


def resize_bilinear_nhwc(logits, out, crop=None):
    """logits f32 NHWC [B,h,w,C] -> out f32 NHWC [B,oh,ow,C]; crop = (y0, x0, ch, cw) source window (default: all)."""
    _chk(logits, f32, "logits"); _chk(out, f32, "out")
    B, h, w, Cc = logits.shape
    y0, x0, ch, cw = crop if crop is not None else (0, 0, h, w)
    L.check(L.lib().ldm_resize_bilinear_nhwc(_p(logits), _p(out), B, h, w, Cc, y0, x0, ch, cw, out.shape[1],
                                             out.shape[2], _stream()), "ldm_resize_bilinear_nhwc")
    return out


def segment_filter(ids, counts, cleaned, *, count_th, overlap_th, ignore_label):
    _chk(ids, i32, "ids"); _chk(counts, i32, "counts"); _chk(cleaned, i32, "cleaned")
    B = ids.shape[0]
    L.check(L.lib().ldm_segment_filter(_p(ids), _p(counts), _p(cleaned), B, ids.numel() // B, counts.shape[-1],
                                       count_th, float(overlap_th), ignore_label, _stream()), "ldm_segment_filter")
    return cleaned


def decode_bitmap(x, ids, quirk31=True):
    _chk(x, f32, "x"); _chk(ids, i32, "ids")
    B, n = x.shape[0], x.shape[1]
    L.check(L.lib().ldm_decode_bitmap(_p(x), _p(ids), B, n, x.numel() // (B * n), int(quirk31), _stream()),
            "ldm_decode_bitmap")
    return ids


def encode_bitmap(ids, x, ignore_label, fill):
    _chk(x, f32, "x"); _chk(ids, i32, "ids")
    B, n = x.shape[0], x.shape[1]
    L.check(L.lib().ldm_encode_bitmap(_p(ids), _p(x), B, n, x.numel() // (B * n), ignore_label, fill, _stream()),
            "ldm_encode_bitmap")
    return x


def ccl_label4(sem, target):
    """sem i32 [B,H,W] -> (labels i32 [B,H,W], ncomp i32 [B]) numbered like scipy.ndimage.label (4-connectivity)."""
    _chk(sem, i32, "sem")
    B, H, W = sem.shape
    labels = torch.empty_like(sem)
    ncomp = torch.empty(B, dtype=i32, device=sem.device)
    nbytes = L.lib().ldm_ccl_scratch_bytes(B, H, W)
    scratch = torch.empty(nbytes // 4, dtype=i32, device=sem.device)
    L.check(L.lib().ldm_ccl_label4(_p(sem), target, _p(labels), _p(ncomp), _p(scratch), B, H, W, _stream()),
            "ldm_ccl_label4")
    return labels, ncomp


def _decode_hist_table(k, c):
    """One hash table (uint64 keys, int32 counts as numpy arrays) -> (a, b, counts) int64 arrays sorted by (a, b)."""
    import numpy as np
    used = k != np.uint64(L.HASH_EMPTY)
    k, c = k[used], c[used].astype(np.int64)
    av = (k >> np.uint64(32)).astype(np.uint32).view(np.int32).astype(np.int64)
    bv = (k & np.uint64(0xFFFFFFFF)).astype(np.uint32).view(np.int32).astype(np.int64)
    order = np.lexsort((bv, av))
    return av[order], bv[order], c[order]


def joint_hist_batch(a, b, n_tables, n_per_table, stride, capacity=1 << 11):
    """`n_tables` joint histograms in ONE launch and ONE device->host copy: table t counts the pairs
    (a.flat[t * stride + j], b.flat[t * stride + j]), j < n_per_table (all images of a batch: stride = n_per_table =
    H * W; sliding windows of k frames: stride = H * W, n_per_table = k * H * W). Returns a list of (a_ids, b_ids,
    counts) int64 numpy triples sorted by (a, b). The tables start at 2 048 slots and grow 8x when one fills up."""
    _chk(a, i32, "a"); _chk(b, i32, "b")
    if (n_tables - 1) * stride + n_per_table > a.numel() or a.numel() != b.numel():
        raise L.LdmError("joint_hist_batch: the last table reads past the end of the maps")
    dev = a.device
    keys = torch.empty((n_tables, capacity), dtype=torch.int64, device=dev)
    counts = torch.empty((n_tables, capacity), dtype=i32, device=dev)
    ovf = torch.empty(n_tables, dtype=i32, device=dev)
    L.check(L.lib().ldm_joint_hist_batch(_p(a), _p(b), n_per_table, stride, n_tables, _p(keys), _p(counts), capacity,
                                         _p(ovf), _stream()), "ldm_joint_hist_batch")
    # one packed transfer: [keys as 2 x int32 | counts | overflow]
    packed = torch.cat([keys.view(i32).reshape(-1), counts.reshape(-1), ovf]).cpu().numpy()
    nk = n_tables * capacity
    if packed[3 * nk:].any():
        if capacity >= 1 << 23:
            raise L.LdmError("joint_hist_batch: more than 2^23 distinct id pairs in one table")
        return joint_hist_batch(a, b, n_tables, n_per_table, stride, capacity * 8)
    import numpy as np
    k = packed[:2 * nk].view(np.uint64).reshape(n_tables, capacity)
    c = packed[2 * nk:3 * nk].reshape(n_tables, capacity)
    return [_decode_hist_table(k[t], c[t]) for t in range(n_tables)]


def city_pan_maps(pred_seg, gt_sem, thing_slots, n_things, ignore_label=0, max_ins=1 << 20):
    """Batched cityscapes_pap_eval.py:66-110: pred_seg / gt_sem i32 [B,H,W] -> (pred_pan, gt_pan) i32 [B,H,W].
    thing_slots: int8 [2, 256] device tensor (see include/ldmseg_b200.h)."""
    _chk(pred_seg, i32, "pred_seg"); _chk(gt_sem, i32, "gt_sem"); _chk(thing_slots, torch.int8, "thing_slots")
    if pred_seg.shape != gt_sem.shape or pred_seg.dim() != 3:
        raise L.LdmError(f"city_pan_maps: prediction {tuple(pred_seg.shape)} vs ground truth {tuple(gt_sem.shape)}")
    B, H, W = pred_seg.shape
    pred_pan, gt_pan = torch.empty_like(pred_seg), torch.empty_like(gt_sem)
    nbytes = L.lib().ldm_city_pan_scratch_bytes(B, H, W, n_things)
    scratch = torch.empty(nbytes // 4, dtype=i32, device=pred_seg.device)
    L.check(L.lib().ldm_city_pan_maps(_p(pred_seg), _p(gt_sem), _p(pred_pan), _p(gt_pan), _p(thing_slots), n_things,
                                      ignore_label, max_ins, _p(scratch), B, H, W, _stream()), "ldm_city_pan_maps")
    return pred_pan, gt_pan


def joint_hist(a, b, capacity=1 << 10):
    """Counts of distinct (a[i], b[i]) pairs. Returns (a_ids, b_ids, counts) as int64 numpy arrays sorted by
    (a, b) -- i.e. the np.unique(a*offset+b, return_counts=True) of the reference in ascending key order.
    The table starts small (a frame has a few hundred distinct id pairs; the whole table is read back: 12 KB at 1 024
    slots) and is retried 16x larger when it fills up."""
    import numpy as np
    _chk(a, i32, "a"); _chk(b, i32, "b")
    keys = torch.empty(capacity, dtype=torch.int64, device=a.device)
    counts = torch.empty(capacity, dtype=i32, device=a.device)
    ovf = torch.empty(1, dtype=i32, device=a.device)
    L.check(L.lib().ldm_joint_hist(_p(a), _p(b), a.numel(), _p(keys), _p(counts), capacity, _p(ovf), _stream()),
            "ldm_joint_hist")
    if int(ovf.item()) != 0:
        if capacity >= 1 << 24:
            raise L.LdmError("joint_hist: more than 2^24 distinct id pairs")
        return joint_hist(a, b, capacity * 16)
    k = keys.cpu().numpy().view(np.uint64)
    c = counts.cpu().numpy()
    used = k != np.uint64(L.HASH_EMPTY)
    k, c = k[used], c[used].astype(np.int64)
    av = (k >> np.uint64(32)).astype(np.uint32).view(np.int32).astype(np.int64)
    bv = (k & np.uint64(0xFFFFFFFF)).astype(np.uint32).view(np.int32).astype(np.int64)
    order = np.lexsort((bv, av))
    return av[order], bv[order], c[order]


def pan_combine(cat, ins, max_ins, pan=None):
    """pan = cat * max_ins + ins on int32 device maps (eval_dvpq.py:108-121)."""
    _chk(cat, i32, "cat"); _chk(ins, i32, "ins")
    if pan is None:
        pan = torch.empty_like(cat)
    _chk(pan, i32, "pan")
    L.check(L.lib().ldm_pan_combine(_p(cat), _p(ins), max_ins, _p(pan), cat.numel(), _stream()), "ldm_pan_combine")
    return pan


def pan_insert(sem, labels, target, max_ins, pan):
    _chk(sem, i32, "sem"); _chk(labels, i32, "labels"); _chk(pan, i32, "pan")
    L.check(L.lib().ldm_pan_insert(_p(sem), _p(labels), target, max_ins, _p(pan), sem.numel(), _stream()),
            "ldm_pan_insert")
    return pan


def id_mask(x, a, va, b=None, vb=0, fill=-1):
    _chk(x, i32, "x"); _chk(a, i32, "a"); _chk(b, i32, "b")
    L.check(L.lib().ldm_id_mask(_p(x), _p(a), va, _p(b), vb, fill, x.numel(), _stream()), "ldm_id_mask")
    return x


def depth_mask_pred(pred, depth_pred, depth_gt, elem_bits, thres, fill):
    """In place on pred (int32 [H, Wp]): ids of the pixels whose abs-rel depth error exceeds thres become `fill`
    (eval_dvpq.py:123-145). depth maps: int32 [H, Wd], Wd <= Wp. Returns abs_rel (float, mean over depth_gt > 0)."""
    _chk(pred, i32, "pred"); _chk(depth_pred, i32, "depth_pred"); _chk(depth_gt, i32, "depth_gt")
    H, Wd = depth_gt.shape
    if depth_pred.shape != depth_gt.shape or pred.shape[0] != H or pred.shape[1] < Wd:
        raise L.LdmError(f"depth_mask_pred: shapes pred={tuple(pred.shape)} depth={tuple(depth_pred.shape)}/{tuple(depth_gt.shape)}")
    nb = 64
    psum = torch.empty(nb, dtype=torch.float64, device=pred.device)
    pcnt = torch.empty(nb, dtype=torch.int64, device=pred.device)
    L.check(L.lib().ldm_depth_mask_pred(_p(pred), pred.stride(0), _p(depth_pred), _p(depth_gt), H, Wd, elem_bits, float(thres),
                                        fill, _p(psum), _p(pcnt), nb, _stream()), "ldm_depth_mask_pred")
    s, c = psum.cpu().numpy(), pcnt.cpu().numpy()
    tot, n = 0.0, 0
    for a, b in zip(s.tolist(), c.tolist()):  # fixed order
        tot += a
        n += b
    return tot / n if n else float("nan")
