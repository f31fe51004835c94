"""Every ops.gemm launch of the production plans, checked against the fp64 reference of tests/gemm_plan_walk.py at its
own shape and the configuration the cost model selected for it.

Per launch: the elementwise bound and the per-tile rms criterion on every output, the write-set (every element written,
guards around the output intact, QKV padding / ones row / zero rows kept, every row_stats entry written), and a repeat
of the launch into guarded scratch outputs that must equal the production output bit for bit (split-K: with the
workspace filled with NaN first). Per UNet plan: the output of the walk (one launch at a time, synchronised) equals an
eager back-to-back run and a CUDA-graph replay bit for bit, which a read of a producer's output before it is complete
(programmatic dependent launch) would break. On a 148-SM B200, the selected configurations must equal
tests/golden/gemm_launch_configs.json (tools/gemm_launch_configs.py regenerates it)."""
import json
import os
import time

import pytest
import torch

import gemm_plan_walk as W
import gpu_kernel_checks as GK

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "gemm_launch_configs.json")
GUARD = 64 << 10              # bytes of NaN sentinel on each side of a scratch output (a multiple of 1 KB: TMA alignment)
WORST = {}                    # (epilogue mode | "fp32") -> [worst elementwise ratio, worst tile ratio]


def _guarded(t, fill=None):
    """A scratch copy of `t` inside a larger allocation whose margins hold 0xFF bytes (NaN in bf16 and fp32). The copy
    holds `fill` (a tensor like t) or 0xFF bytes. Returns (raw bytes, view)."""
    n = t.numel() * t.element_size()
    raw = torch.full((2 * GUARD + (n + 1023) // 1024 * 1024,), 0xFF, dtype=torch.uint8, device=t.device)
    view = raw[GUARD:GUARD + n].view(t.dtype).view(t.shape)
    if fill is not None:
        view.copy_(fill)
    return raw, view


def _bytes(t):
    return t.reshape(-1).view(torch.uint8)


def _guards_intact(raw, n):
    return bool((raw[:GUARD] == 0xFF).all()) and bool((raw[GUARD + n:] == 0xFF).all())


def _region(name, d, seq):
    """The written region of a QKV buffer."""
    return (slice(None), slice(None), slice(0, d)) if name != "vt" else (slice(None), slice(0, d), slice(0, seq))


class Checker:
    def __init__(self, plan):
        from video_latent_diffusion_panoptic_segmentation_b200 import ops
        self.ops, self.gemm, self.plan, self.recs = ops, ops.gemm, plan, []

    def __call__(self, a, k, name):
        ops = self.ops
        c = W.snapshot(a, k)
        self.gemm(*a, **k)
        bn, pair, split = ops.gemm_last_config()
        torch.cuda.synchronize()
        desc = W.describe(a, k)
        rec = dict(name=name, desc=desc, block_n=bn, pair=pair, split=split)
        where = f"{self.plan} / {name}: block_n={bn} pair={pair} split={split} {desc}"
        for key in ("residual", "rowbias", "a2"):
            assert c[key] is None or torch.equal(k[key], c[key]), f"{where}: the launch changed its {key} (aliasing)"
        assert torch.equal(a[0], c["a1"]), f"{where}: the launch changed its a1 (aliasing)"
        outs = W.gemm_reference(c)
        q = k.get("qkv")
        got = {"out": a[2]} if q is None else {
            n: q[n][_region(n, q["head_dim"], q["seq"])] for n in ("q", "k", "vt") if n in outs}
        for key, o in outs.items():
            g = got[key].reshape(o.ref.shape)
            res = GK._bound_stats(g, o.ref, o.mag_eff(), f"{where} [{key}]", W.U if o.bf16_out else 2.0 ** -24, o.a,
                                  where=lambda i: {"index": i, "tile_128": i[0] // 128 if len(i) else None})
            tw = 0.0
            if o.bf16_out:
                tw, (ti, tj) = W.tile_stats(g, o, key, bn)
                assert tw <= 1.0, (f"{where} [{key}]: tile (rows {ti * 128}..{ti * 128 + 127}, columns {tj * bn}.."
                                   f"{tj * bn + bn - 1}) rms error {tw:.2f} x its bound (kappa {W.KAPPA})")
            rec.setdefault("worst", {})[key] = (res["worst_ratio"], tw)
        if k.get("row_stats") is not None:
            ref, bound = W.row_stats_ref(a[2], a[2].numel() // a[2].shape[-1])
            st = k["row_stats"].double()
            assert torch.isfinite(st).all(), f"{where}: row_stats has unwritten entries"
            assert ((st - ref).abs() <= bound).all(), f"{where}: row_stats differ from the sums of the bf16 output"
        if q is not None:   # padding columns, the V^T ones row and zero rows, columns past seq: as before the launch
            for n, before in c["qkv_before"].items():
                keep = torch.ones_like(before, dtype=torch.bool)
                keep[_region(n, q["head_dim"], q["seq"])] = False
                assert torch.equal(q[n][keep], before[keep]), f"{where}: {n} changed outside the written region"
        self._repeat(a, k, c, rec, where)
        self.recs.append(rec)

    def _repeat(self, a, k, c, rec, where):
        """The same launch into guarded scratch outputs: all written, guards intact, bit-identical to production."""
        ops = self.ops
        a2, k2, checks = list(a), dict(k), []
        q = k.get("qkv")
        if q is None:
            raw, view = _guarded(a[2])
            a2[2] = view
            checks.append(("out", raw, a[2]))
        else:
            q2 = dict(q)
            for n, before in c["qkv_before"].items():
                raw, view = _guarded(before, before)
                view[_region(n, q["head_dim"], q["seq"])] = float("nan")
                q2[n] = view
                checks.append((n, raw, q[n]))
            k2["qkv"] = q2
        if k.get("row_stats") is not None:
            raw, view = _guarded(k["row_stats"])
            k2["row_stats"] = view
            checks.append(("row_stats", raw, k["row_stats"]))
        if rec["split"] > 1:
            ops._splitk_ws(a[0].device).fill_(0xFF)      # a fix-up that reads a slice nobody wrote sees NaN
        self.gemm(*a2, **k2)
        cfg = ops.gemm_last_config()
        torch.cuda.synchronize()
        assert cfg == (rec["block_n"], rec["pair"], rec["split"]), f"{where}: the repeat selected {cfg}"
        for n, raw, prod in checks:
            nb = prod.numel() * prod.element_size()
            assert _guards_intact(raw, nb), f"{where}: the launch wrote outside {n}"
            same = torch.equal(raw[GUARD:GUARD + nb], _bytes(prod))
            assert same, f"{where}: {n} of the repeat differs from production (unwritten elements or not reproducible)"


def _golden():
    with open(GOLDEN) as f:
        return json.load(f)


WALKS = dict(W.plan_walks())
CONFIGS = {}                  # plan -> the config walk's records (test_plan_gemm_launches fills it)


@pytest.mark.gpu
@pytest.mark.parametrize("plan", list(WALKS))
def test_plan_gemm_launches(plan):
    t0 = time.time()
    builder = WALKS[plan]
    cfg = CONFIGS[plan] = W.config_walk(builder)
    if torch.cuda.get_device_properties(0).multi_processor_count == 148:
        want = _golden()[plan].split()
        moved = [(r["name"], r["desc"], w_, W.config_code(r)) for r, w_ in zip(cfg, want) if W.config_code(r) != w_]
        assert len(want) == len(cfg) and not moved, \
            f"{plan}: selected configurations differ from {os.path.basename(GOLDEN)} ({len(want)} pinned launches, " \
            f"{len(cfg)} walked); (launch, descriptor, pinned, selected): {moved[:10]}"
    chk = Checker(plan)
    res = builder(chk)
    assert len(chk.recs) == len(cfg), f"{plan}: {len(chk.recs)} checked launches, {len(cfg)} in the config walk"
    for r, c in zip(chk.recs, cfg):
        assert (r["name"], r["block_n"], r["pair"], r["split"]) == (c["name"], c["block_n"], c["pair"], c["split"])
        for key, (e, t) in r["worst"].items():
            mode = "fp32" if r["desc"]["flags"] & (W.OUT_F32 | W.OUT_NCHW_F32) else c["epilogue"]
            w_ = WORST.setdefault(mode, [0.0, 0.0, 0])
            w_[0], w_[1], w_[2] = max(w_[0], e), max(w_[1], t), w_[2] + 1
    if "st" in res:   # plan-level ordering: eager back to back and a graph replay give the walk's output bit for bit
        unet, st, walk_out = res["unet"], res["st"], res["out"]
        st.out.fill_(float("nan"))
        unet._run_plan(st)
        torch.cuda.synchronize()
        assert torch.equal(st.out, walk_out), f"{plan}: an eager run differs from the launch-by-launch walk"
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            unet._run_plan(st)
        st.out.fill_(float("nan"))
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(st.out, walk_out), f"{plan}: a CUDA-graph replay differs from the launch-by-launch walk"
        del g
    print(f"\nGEMM_WALK {json.dumps(dict(plan=plan, launches=len(chk.recs), seconds=round(time.time() - t0, 1), worst=WORST))}")


# what the walk must reach, so that a selection change that drops a path says so
PATHS = {
    "staged epilogue, CTA pair": lambda r: r["epilogue"] == "staged" and r["pair"],
    "staged epilogue, single CTA": lambda r: r["epilogue"] == "staged" and not r["pair"],
    "split-K on a CTA pair": lambda r: r["split"] > 1 and r["pair"],
    "QKV TMA stores, whole-image tiles": lambda r: _qkv_tma(r) and not W.qkv_straddles(r["desc"]),
    "QKV TMA stores, tiles straddling two images": lambda r: _qkv_tma(r) and W.qkv_straddles(r["desc"]),
    "up2": lambda r: r["desc"].get("up2", False),
    "gather + conv up-sampling": lambda r: "upsamplers.0.conv" in r["name"] and not r["desc"].get("up2"),
    "stride 2, pad 0": lambda r: r["desc"].get("a_stride") == 2 and r["desc"]["a_pad"] == 0,
    "stride 2, pad 1": lambda r: r["desc"].get("a_stride") == 2 and r["desc"]["a_pad"] == 1,
    "GEGLU": lambda r: r["epilogue"] == "geglu",
    "GEGLU with the LayerNorm fold": lambda r: r["epilogue"] == "geglu_ln",
    "QKV with the LayerNorm fold": lambda r: r["epilogue"] == "qkv_ln",
    "ConvT + LayerNorm2d + SiLU": lambda r: r["epilogue"] == "convt",
    "NCHW fp32": lambda r: bool(r["desc"]["flags"] & W.OUT_NCHW_F32),
}


def _qkv_tma(r):
    """The QKV launches that leave through TMA stores: block_n 160, single CTA, K <= 384, seq >= 128 (gemm_tc.cu)."""
    q = r["desc"].get("qkv")
    return (q is not None and r["epilogue"] in ("qkv", "qkv_ln") and r["block_n"] == 160 and not r["pair"] and
            r["desc"]["K"] <= 384 and q["seq"] >= 128 and 160 % q["d"] == 0)


@pytest.mark.gpu
def test_plans_reach_every_path():
    for plan, builder in WALKS.items():   # (plans whose launch check was not run are walked here)
        if plan not in CONFIGS:
            CONFIGS[plan] = W.config_walk(builder)
    recs = [r for plan in CONFIGS.values() for r in plan]
    missing = [p for p, f in PATHS.items() if not any(f(r) for r in recs)]
    assert not missing, f"the production plans no longer reach: {missing}"


def test_pinned_configs_list_every_plan():
    assert sorted(_golden()) == sorted(WALKS), f"{os.path.basename(GOLDEN)} does not list every walked plan"
