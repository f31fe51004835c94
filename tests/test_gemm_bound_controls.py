"""Sensitivity of the contraction comparator of tests/gemm_plan_walk.py (CPU, fp64, no GPU needed).

The plan walk (tests/test_gemm_plan_launches_gpu.py) passes a launch when every output stays within a quarter of the
elementwise bound and every 128-row x block_n tile within its rms bound. These controls show, on a few hundred output
rows at the production K of each class, that the same comparator flags a reference with one small, plausible kernel
bug, and passes the unmutated reference rounded to bf16 as the kernel rounds it."""
import pytest
import torch

import gemm_plan_walk as W
import gpu_kernel_checks as GK

bf16, f64 = torch.bfloat16, torch.float64
ROWS, BN = 256, 160       # two 128-row tiles, one 160-column tile (the block_n of the 320-wide layers)

# production K per class: (K, taps, c1, c2) -- the L3 concat conv (2560 = 1280 + 1280 channels), the 1920-channel
# concat conv, the 1280-channel conv, ff2 of L2 / L3, the level-0 conv and pointwise GEMMs, the RGB VAE's P V
K_CLASSES = [(23040, 9, 1280, 1280), (17280, 9, 1280, 640), (11520, 9, 1280, 0), (5120, 1, 5120, 0),
             (2880, 9, 320, 0), (320, 1, 320, 0), (7488, 1, 7488, 0)]


def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _operands(K, N=BN, rows=ROWS, seed=0):
    g = _gen(seed)
    a = torch.randn((rows, K), generator=g).to(bf16)
    w = (torch.randn((N, K), generator=g) * K ** -0.5).to(bf16)
    bias = torch.randn(N, generator=g)
    res = torch.randn((rows, N), generator=g).to(bf16)
    return a, w, bias, res


def _ref(a, w, **k):
    c = dict(a1=a, w=w, flags=0, taps=1)
    c.update(k)
    return W.gemm_reference(c)


def _flagged(got, o, key="out"):
    """What the plan walk rejects: an element above the elementwise bound or a tile above its rms bound."""
    if W.elementwise_ratio(got, o).max().item() > 1.0:
        return True
    return o.bf16_out and W.tile_stats(got, o, key, BN)[0] > 1.0


def _passes(o, key="out"):
    got = o.ref.to(bf16)
    return (W.elementwise_ratio(got, o).max().item() <= GK.BOUND_HEADROOM and
            (not o.bf16_out or W.tile_stats(got, o, key, BN)[0] <= 1.0))


def _mm(a, w):
    return a.to(f64) @ w.to(f64).t()


@pytest.mark.parametrize("K,taps,c1,c2", K_CLASSES)
def test_dropped_k_block(K, taps, c1, c2):
    """One 64-wide K block missing from every output of the launch: the first, a middle one, the last, the first block
    of the second tap, and the first block of a2 (concat sources)."""
    a, w, bias, _ = _operands(K, seed=K)
    o = _ref(a, w, bias=bias)["out"]
    assert _passes(o)
    ktap = c1 + c2
    starts = {0, (K // 2) // 64 * 64, K - 64}
    if taps > 1:
        starts.add(ktap)
    if c2:
        starts.add(c1)
    for k0 in sorted(starts):
        keep = torch.cat([torch.arange(k0), torch.arange(k0 + 64, K)])
        got = (_mm(a[:, keep], w[:, keep]) + bias.double()).to(bf16)
        assert _flagged(got, o), f"K={K}: the K block at {k0} dropped is not flagged"


def test_dropped_block_needs_the_tile_criterion(monkeypatch):
    """With the tile criterion loosened (kappa = 1e6), the elementwise bound alone misses a dropped block at K = 23 040:
    the tile criterion is what constrains long-K launches."""
    K = 23040
    a, w, bias, _ = _operands(K, seed=K)
    o = _ref(a, w, bias=bias)["out"]
    k0 = (K // 2) // 64 * 64
    keep = torch.cat([torch.arange(k0), torch.arange(k0 + 64, K)])
    got = (_mm(a[:, keep], w[:, keep]) + bias.double()).to(bf16)
    assert _flagged(got, o)
    monkeypatch.setattr(W, "KAPPA", 1e6)
    assert not _flagged(got, o)


@pytest.mark.parametrize("K,split", [(23040, 3), (11520, 3), (5120, 2)])
def test_split_k_slice(K, split):
    """Split-K: the fix-up of ONE tile (rows 128..255) misses one slice's partial, or adds it twice."""
    a, w, bias, res = _operands(K, seed=K + 1)
    o = _ref(a, w, bias=bias, residual=res)["out"]
    assert _passes(o)
    s0, s1 = K // split, 2 * K // split          # the middle slice
    part = _mm(a[128:, s0:s1], w[:, s0:s1])
    full = _mm(a, w) + bias.double() + res.double()
    for sign in (-1.0, 1.0):
        m = full.clone()
        m[128:] += sign * part
        assert _flagged(m.to(bf16), o), f"K={K}: split slice {'dropped' if sign < 0 else 'counted twice'} not flagged"


# one-line epilogue bugs of a launch with bias and residual, built from the exact fp64 pieces (acc, bias, residual, ref)
MUTATIONS = {
    "residual added twice": lambda acc, b, r, ref: acc + b + 2 * r,
    "columns 48..63 without their bias": lambda acc, b, r, ref: acc + b * (torch.arange(b.numel()) // 16 != 3) + r,
    "rows of tile 1 shifted by one": lambda acc, b, r, ref: torch.cat([ref[:128], ref[129:], ref[-1:]]),
}


@pytest.mark.parametrize("mutation", list(MUTATIONS))
@pytest.mark.parametrize("K", [23040, 5120, 2880, 320])
def test_output_mutations(K, mutation):
    a, w, bias, res = _operands(K, seed=K + 2)
    o = _ref(a, w, bias=bias, residual=res)["out"]
    assert _passes(o)
    got = MUTATIONS[mutation](_mm(a, w), bias.double(), res.double(), o.ref)
    assert _flagged(got.to(bf16), o), f"K={K}: {mutation} is not flagged"


def _conv_flat(x, w, H, Wd, halo_bug):
    """3x3 convolution (padding 1) of one image x [H*W, C] in fp64. halo_bug: a tap left or right of the image reads
    the neighbouring row's pixel (flattened index +-1) instead of the zero padding."""
    HW, C = x.shape
    idx = torch.arange(HW)
    yy, xx = idx // Wd, idx % Wd
    out = torch.zeros((HW, w.shape[0]), dtype=f64)
    for ky in range(3):
        for kx in range(3):
            p = idx + (ky - 1) * Wd + (kx - 1)
            ok = (p >= 0) & (p < HW)
            if not halo_bug:
                ok &= (xx + kx - 1 >= 0) & (xx + kx - 1 < Wd) & (yy + ky - 1 >= 0) & (yy + ky - 1 < H)
            t = 3 * ky + kx
            src = torch.zeros((HW, C), dtype=f64)
            src[ok] = x[p[ok]].to(f64)
            out += src @ w[:, t * C:(t + 1) * C].to(f64).t()
    return out


@pytest.mark.parametrize("H,Wd,c1,c2", [(6, 20, 1280, 1280), (12, 39, 1280, 640), (48, 156, 320, 0)])
def test_halo_reads_neighbour_row(H, Wd, c1, c2):
    """3x3 conv at the production level shapes (one image; the 48x156 level: its first 312 pixels)."""
    g = _gen(H)
    C = c1 + c2
    rows = min(H, 3) * Wd if H > 12 else H * Wd
    Hc = rows // Wd
    x1 = torch.randn((1, Hc, Wd, c1), generator=g).to(bf16)
    x2 = torch.randn((1, Hc, Wd, c2), generator=g).to(bf16) if c2 else None
    w = (torch.randn((BN, 9 * C), generator=g) * (9 * C) ** -0.5).to(bf16)
    o = W.gemm_reference(dict(a1=x1, a2=x2, w=w, flags=0, taps=9))["out"]
    assert _passes(o)
    x = x1 if x2 is None else torch.cat([x1, x2], -1)
    exact = _conv_flat(x.view(-1, C), w, Hc, Wd, False)
    assert torch.allclose(exact, o.ref.view(-1, BN), rtol=1e-12, atol=1e-9)   # the two references agree
    bug = _conv_flat(x.view(-1, C), w, Hc, Wd, True)
    assert _flagged(bug.to(bf16).view(o.ref.shape), o)


@pytest.mark.parametrize("K", [1280, 320])
def test_geglu_blocks_offset(K):
    """GEGLU: the gate of output block j read from the next 16-row block (the value / gate interleave off by one)."""
    g = _gen(K + 4)
    N = 2 * BN
    a = torch.randn((ROWS, K), generator=g).to(bf16)
    w = (torch.randn((N, K), generator=g) * K ** -0.5).to(bf16)
    bias = torch.randn(N, generator=g)
    o = _ref(a, w, bias=bias, flags=W.GEGLU)["out"]
    assert _passes(o)
    h = (_mm(a, w) + bias.double()).view(ROWS, N // 32, 2, 16)
    v, gt = h[:, :, 0], h[:, :, 1].roll(-1, dims=1)
    got = (v * W._gelu(gt)).reshape(ROWS, N // 2)
    assert _flagged(got.to(bf16), o)


def test_qkv_head_columns_shifted():
    """The QKV split at level 0 (8 heads of 40, K = 320, 256 tokens of one image): head 3's q columns read one column
    to the right (channel j of the head gets j + 1; the last reads the next head's first)."""
    heads, d, seq, K = 8, 40, ROWS, 320
    C = heads * d
    g = _gen(5)
    a = torch.randn((seq, K), generator=g).to(bf16)
    w = (torch.randn((3 * C, K), generator=g) * K ** -0.5).to(bf16)
    qkv = dict(heads=heads, head_dim=d, dpad=64, seq=seq, seq_pad=seq)
    outs = _ref(a, w, flags=W.QKV_SPLIT, qkv=qkv)
    o = outs["q"]
    assert _passes(o, "q") and _passes(outs["vt"], "vt")
    full = _mm(a, w)
    m = o.ref.clone()
    m[3] = full[:, 3 * d + 1:4 * d + 1]
    assert _flagged(m.to(bf16), o, "q")


@pytest.mark.parametrize("flags", [W.OUT_F32, W.SILU, W.GEGLU])
def test_unmutated_modes_pass(flags):
    """fp32 output, SiLU and GEGLU at K = 2880 / 1280: the unmutated reference, rounded as the kernel rounds its output,
    passes both criteria."""
    K = 2880 if flags != W.GEGLU else 1280
    a, w, bias, _ = _operands(K, N=2 * BN, seed=K + 7)
    o = _ref(a, w, bias=bias, flags=flags)["out"]
    got = o.ref.float() if not o.bf16_out else o.ref.to(bf16)
    assert W.elementwise_ratio(got, o).max().item() <= GK.BOUND_HEADROOM
    if o.bf16_out:
        assert W.tile_stats(got, o, "out", BN)[0] <= 1.0


def test_f32_output_dropped_block():
    """fp32 outputs have no tile criterion: the elementwise bound alone must flag a dropped block at their K (the UNet's
    conv_out, K = 2 880)."""
    K = 2880
    a, w, bias, _ = _operands(K, N=8, seed=K + 8)
    o = _ref(a, w, bias=bias, flags=W.OUT_F32)["out"]
    keep = torch.cat([torch.arange(1408), torch.arange(1472, K)])
    got = (_mm(a[:, keep], w[:, keep]) + bias.double()).float()
    assert _flagged(got, o)
