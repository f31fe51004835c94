"""Sensitivity of the bound comparator of gpu_kernel_checks.py (CPU, no GPU needed).

The GPU checks pass when a kernel stays within a quarter of |got - ref| <= r |ref| + a mag. These controls show that the
same comparator, on the same data and at the largest shape of each class in the plans, flags a reference with one
small, plausible bug -- and passes the unmutated reference rounded to bf16, as a kernel would write it."""
import math

import pytest
import torch

import gpu_kernel_checks as K

bf16 = torch.bfloat16


def _flagged(got, ref, mag, a):
    return K.bound_ratio(got, ref, mag, K.U_BF16, a).max().item() > 1.0


def _passes(ref, mag, a):
    return K.bound_ratio(ref.to(bf16), ref, mag, K.U_BF16, a).max().item() <= K.BOUND_HEADROOM


# (head_dim, tokens, key block) of the largest self-attention of each head width; data of check_attention_bound
@pytest.mark.parametrize("d,seq,blk", [(40, 7488, 96), (80, 1872, 64), (160, 468, 64)])
def test_attention_controls(d, seq, blk):
    q, k, v = (t[:1] for t in K.attn_random_inputs(seq, seq, d, 2, 4.0, 300 + d))   # head 0 of the GPU check
    scale = d ** -0.5
    ref, mag = K.attn_ref(q, k, v, scale)
    assert _passes(ref, mag, K.A_ATTN)
    j0 = (seq // 2) // blk * blk                                  # one key block dropped
    keep = torch.cat([torch.arange(j0), torch.arange(j0 + blk, seq)])
    assert _flagged(K.attn_ref(q, k[:, keep], v[:, keep], scale)[0].to(bf16), ref, mag, K.A_ATTN)
    vm = v.clone()                                                # the ones row (row sums) read as a data channel
    vm[:, :, d - 1] = 1.0
    assert _flagged(K.attn_ref(q, k, vm, scale)[0].to(bf16), ref, mag, K.A_ATTN)


@pytest.mark.parametrize("kv", K.EDGE_KV)
@pytest.mark.parametrize("margin", [7.0, 20.0, 40.0, 100.0])
def test_needle_inputs(kv, margin):
    """The needle is each row's unique maximum, at least `margin` log2 units above every other key, and the positions
    cover both sides of every boundary inside the sequence."""
    d = 40
    S = min(kv, 300)
    q, k, v, tgt = K.needle_inputs(S, kv, d, margin)
    s = (q.double() @ k.double().transpose(1, 2)) * d ** -0.5 * math.log2(math.e)
    top = s.max(-1)
    assert torch.equal(top.indices, tgt)
    if kv > 1:
        second = s.scatter(-1, tgt[..., None], -math.inf).max(-1).values
        assert (top.values - second).min().item() >= 0.99 * margin
    pos = K.needle_positions(kv)
    for b in (0, 47, 48, 63, 64, 95, 96, kv - 1):
        assert b >= kv or b in pos


def _group_stats(x, groups, eps):
    B, HW, C = x.shape
    xg = x.double().view(B, HW, groups, C // groups)
    mean = xg.mean(dim=(1, 3))
    rstd = 1.0 / torch.sqrt(xg.var(dim=(1, 3), unbiased=False) + eps)
    return mean, rstd


def test_groupnorm_controls():
    """The cooperative-kernel shape (B = 8, 48x156, 320 channels) with the 16-64x means of check_groupnorm_cancel."""
    B, HW, C, G, eps = 8, 7488, 320, 32, 1e-5
    cpg = C // G
    x = K.cancellation_input((B, HW, G, cpg), 60 + B).view(B, HW, C)
    gm = torch.randn(C, generator=torch.Generator().manual_seed(8)) * 0.2 + 1
    bt = torch.randn(C, generator=torch.Generator().manual_seed(9)) * 0.1
    ref, mag = K.norm_ref(x, gm, bt, eps, groups=G)
    assert _passes(ref, mag, K.A_NORM)
    mean, rstd = _group_stats(x, G, eps)
    g = 2                                                         # a 64x group
    cols = slice(g * cpg, (g + 1) * cpg)
    ulp = 2.0 ** (math.floor(math.log2(abs(mean[0, g].item()))) - 7)
    m1 = ref.clone()                                              # its mean off by one bf16 ulp of the mean
    m1[0, :, cols] -= gm[cols].double() * ulp * rstd[0, g]
    assert _flagged(m1.to(bf16), ref, mag, K.A_NORM)
    m2 = ref.clone()                                              # normalised with the neighbouring group's moments
    m2[0, :, cols] = (x[0, :, cols].double() - mean[0, g + 1]) * rstd[0, g + 1] * gm[cols].double() + bt[cols].double()
    assert _flagged(m2.to(bf16), ref, mag, K.A_NORM)


def test_layernorm_controls():
    C, rows, eps = 1280, 2000, 1e-5
    x = K.cancellation_input((rows, 1, 1, C), 70 + C).view(rows, C)
    gm = torch.randn(C, generator=torch.Generator().manual_seed(4)) * 0.2 + 1
    bt = torch.randn(C, generator=torch.Generator().manual_seed(5)) * 0.1
    ref, mag = K.norm_ref(x, gm, bt, eps)
    assert _passes(ref, mag, K.A_NORM)
    xd = x[7].double()
    ulp = 2.0 ** (math.floor(math.log2(abs(xd.mean().item()))) - 7)
    m1 = ref.clone()                                              # one row's mean off by one bf16 ulp of the mean
    m1[7] -= gm.double() * ulp / torch.sqrt(xd.var(unbiased=False) + eps)
    assert _flagged(m1.to(bf16), ref, mag, K.A_NORM)


def test_bound_ratio_edges():
    ref = torch.tensor([0.0, 1.0, 1.0, 2.0], dtype=torch.float64)
    mag = torch.tensor([0.0, 1.0, 1.0, 2.0], dtype=torch.float64)
    got = torch.tensor([0.0, float("nan"), 1.0, float("inf")])
    r = K.bound_ratio(got, ref, mag, K.U_BF16, K.A_ATTN)
    assert r[0] == 0 and math.isinf(r[1]) and r[2] == 0 and math.isinf(r[3])
    assert math.isinf(K.bound_ratio(torch.tensor([1e-30]), torch.zeros(1), torch.zeros(1), K.U_BF16, K.A_ATTN)[0])
    with pytest.raises(AssertionError, match="first_bad"):
        K._bound_stats(got, ref, mag, "edges", K.U_BF16, K.A_ATTN)
