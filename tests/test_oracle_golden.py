"""CPU: the oracle restatements (oracle/) against the golden fixtures that tests/golden/make_golden.py produced by
running the REAL reference code, plus the reference's own sample_outputs/ bit-codec vector and hand-computed cases."""
import json
import os

import numpy as np
import torch

from oracle import eval_oracle as EO
from oracle import ldmseg_oracle as LO
from synth import city_case, vpq_case

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GOLD = json.load(open(os.path.join(G, "golden.json")))


def test_ddim_timesteps_and_schedule():
    s = LO.DDIMOracle()
    for T in (10, 50):
        s.set_timesteps_inference(T)
        assert s.timesteps.tolist() == GOLD["scheduler"][f"timesteps_{T}"]
    assert GOLD["scheduler"]["timesteps_50"][0] == 999 and GOLD["scheduler"]["timesteps_50"][-1] == 19
    want = GOLD["scheduler"]["alphas_cumprod_0_19_999"]
    assert [float(s.alphas_cumprod[i]) for i in (0, 19, 999)] == want
    assert want[0] == 0.9991499781608582 and want[2] == 0.00466009508818388


def test_ddim_step_bit_exact_with_reference():
    z = np.load(os.path.join(G, "ddim_steps.npz"))
    s = LO.DDIMOracle()
    assert np.array_equal(s.alphas_cumprod.numpy(), z["alphas_cumprod"])
    s.set_timesteps_inference(50)
    eps, x = torch.from_numpy(z["eps"]), torch.from_numpy(z["x"])
    for t in (999, 499, 19):  # 19: prev_t < 0 -> final_alpha_cumprod
        prev, x0 = s.step(eps, t, x)
        assert np.array_equal(prev.numpy(), z[f"prev_{t}"])
        assert np.array_equal(x0.numpy(), z[f"x0_{t}"])


def test_ddim_step_clip_bit_exact_with_reference():
    """clip_sample (the reference constructor's default) and use_clipped_model_output, vectors of the real scheduler
    (tests/golden/make_golden_ddim_clip.py). The inputs are wide enough that the clamp bites."""
    z = np.load(os.path.join(G, "ddim_steps_clip.npz"))
    eps, x = torch.from_numpy(z["eps"]), torch.from_numpy(z["x"])
    clipped = 0
    for rng in (1.0, 0.5):
        s = LO.DDIMOracle(clip_sample=True, clip_sample_range=rng)
        s.set_timesteps_inference(50)
        for t in (999, 499, 19):
            for ucm in (False, True):
                prev, x0 = s.step(eps, t, x, use_clipped_model_output=ucm)
                tag = f"r{rng}_t{t}_u{int(ucm)}"
                assert np.array_equal(prev.numpy(), z["prev_" + tag]), tag
                assert np.array_equal(x0.numpy(), z["x0_" + tag]), tag
                clipped += int((np.abs(z["x0_" + tag]) == rng).sum())
    assert clipped > 100


def test_seg_decoder_bit_exact_with_reference():
    z = np.load(os.path.join(G, "seg_decoder_small.npz"))
    cfg = GOLD["seg_decoder_small"]["cfg"]
    dec = LO.SegDecoderOracle(**cfg).eval()
    sd = {k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd.")}
    assert sorted(sd) == GOLD["seg_decoder_small"]["keys"] == sorted(dec.state_dict())
    dec.load_state_dict(sd, strict=True)
    assert dec.interpolation_factor == GOLD["seg_decoder_small"]["interpolation_factor"] == 2
    assert dec.downsample_factor == GOLD["seg_decoder_small"]["downsample_factor"] == 8
    with torch.no_grad():
        lo = dec.decode(torch.from_numpy(z["z"]), interpolate=False)
        hi = dec.decode(torch.from_numpy(z["z"]), interpolate=True)
    assert np.array_equal(lo.numpy(), z["logits_lo"])
    assert np.array_equal(hi.numpy(), z["logits_hi"])


def test_bit_codec_sample_outputs_vector():
    z = np.load(os.path.join(G, "bitmap_sample_outputs.npz"))
    sem = torch.from_numpy(z["semseg"].astype(np.int64))
    bits, ign = LO.encode_bitmap(sem, 16, ignore_label=0, fill_value=0.5)
    assert np.array_equal((bits.numpy() * 255).astype(np.uint8), z["bits_u8"])  # the reference's PNGs
    dec = LO.decode_bitmap(bits)
    assert np.array_equal(dec.numpy(), z["decoded"])
    # non-ignore pixels round-trip except id 31 -> 0 (cityscapes.py:269); ignore pixels (all 0.5) decode to 65535
    ok = (~ign) & (sem != 31)
    assert torch.equal(dec[ok], sem[ok])
    assert int((dec[sem == 31] == 0).sum()) == GOLD["bitmap"]["n_id31"] == 67
    assert bool((dec[ign] == 65535).all())
    assert torch.equal(LO.decode_bitmap(bits, quirk31=False)[sem == 31], sem[sem == 31])


def test_vpq_eval_matches_reference():
    for case in GOLD["vpq"].values():
        pred, gt = vpq_case(case["seed"], case["H"], case["W"])
        for a, b in zip(EO.vpq_stats(pred, gt), case["out"]):
            assert a.tolist() == b  # float64 iou sums bit-exact
        gt64 = (gt // 2 ** 20) * 64 + (gt % 2 ** 20) % 64
        pr64 = (pred // 2 ** 20) * 64 + (pred % 2 ** 20) % 64
        for a, b in zip(EO.vpq_stats(pr64, gt64, max_ins=64, guard_union=True), case["out64"]):
            assert a.tolist() == b


def test_cityscapes_evaluator_matches_reference():
    ev = EO.CityscapesPQOracle()
    for img in GOLD["cityscapes_pq"]["images"]:
        pred, gt = city_case(img["seed"])
        ev.add_image(pred, gt)
        assert (ev.TP, ev.FP, ev.FN) == (img["tp"], img["fp"], img["fn"])
        assert ev.iou_sum == img["iou_sum"]
    res, want = ev.evaluate(), GOLD["cityscapes_pq"]["result"]
    for k in ("pq", "sq", "rq", "tp", "fp", "fn", "iou_sum", "thing_pq", "thing_sq", "thing_rq", "stuff_pq",
              "stuff_sq", "stuff_rq"):
        assert res[k] == want[k], k
    assert {str(c): m for c, m in res["per_class"].items()} == want["per_class"]


def test_vpq_hand_computed_two_segment_image():
    # gt: left half class 3 inst 1, right half class 7 inst 0; pred: class 3 inst 5 covers 3 of 4 left columns +
    # nothing else there (class 9), right half correct.
    M = 2 ** 20
    gt = np.zeros((4, 8), np.int64)
    gt[:, :4], gt[:, 4:] = 3 * M + 1, 7 * M
    pred = np.zeros((4, 8), np.int64)
    pred[:, :3], pred[:, 3], pred[:, 4:] = 3 * M + 5, 9 * M, 7 * M + 2
    iou, tp, fn, fp = EO.vpq_stats(pred, gt)
    assert tp[3] == 1 and iou[3] == 12 / 16 and tp[7] == 1 and iou[7] == 1.0
    assert fn.sum() == 0 and fp[9] == 1 and fp.sum() == 1
    agg = EO.dvpq_aggregate([(iou, tp, fn, fp)])
    assert abs(agg["pq"] - 100 * (0.75 + 1.0) / 19) < 1e-6


def test_merge_hand_computed():
    # 2 classes + ignore: class 0 big and confident, class 1 small (< count_th), class 2 low confidence -> ignore
    C, H, W = 4, 8, 8
    lg = torch.full((C, H, W), -10.0)
    lg[0, :, :5] = 10.0   # 40 px of class 0
    lg[1, :, 5:6] = 10.0  # 8 px of class 1
    lg[2, :, 6:] = -9.9   # 16 px argmax class 2 but softmax max ~ 0.27 < 0.5
    pred, cleaned, kept = LO.logits_to_panoptic(lg, mask_th=0.5, count_th=10, overlap_th=0.5, ignore_label=3)
    assert kept == [0]
    assert (cleaned[:, :5] == 0).all() and (cleaned[:, 5:] == -1).all()
    assert (pred[:, 6:] == 3).all() and (pred[:, 5] == 1).all()


def test_seg_encoder_bit_exact_with_reference():
    """oracle.SegEncoderOracle / SegDecoderOracle == the real GeneralVAESeg encoder, posterior and forward()."""
    import ast
    from oracle import ldmseg_oracle as LO
    z = {k: f[k] for name in ("seg_encoder_small.npz", "seg_encoder_small_part2.npz")
         for f in [np.load(os.path.join(G, name))] for k in f.files}
    cfg = ast.literal_eval(str(z["cfg"]))
    sd = {k[3:]: torch.from_numpy(v) for k, v in z.items() if k.startswith("sd.")}
    enc = LO.SegEncoderOracle(**cfg).eval()
    enc.load_state_dict({k: v for k, v in sd.items() if k.startswith("encoder.")})
    dec = LO.SegDecoderOracle(**cfg).eval()
    dec.load_state_dict({k: v for k, v in sd.items() if k.startswith("decoder.")})
    with torch.no_grad():
        m = enc.encode(torch.from_numpy(z["bits"]))
        mean, _, std = enc.posterior(m)
        fwd = dec.decode(mean, interpolate=False)
    assert np.array_equal(m.numpy(), z["moments"])
    assert np.array_equal(mean.numpy(), z["mode"]) and np.array_equal(std.numpy(), z["std"])
    assert np.array_equal(fwd.numpy(), z["forward"])


def test_evaluator_edge_cases_match_reference():
    """tests/golden/edge_cases.json (real reference outputs, make_golden_edge_cases.py): identical maps, a prediction
    that matches nothing, all-void ground truth, a single pixel, > 1 000 distinct id pairs, IoU exactly 0.5 (strict >),
    an all-void prediction, all-ignore ground truth, 512 single-pixel components, a thing split in two."""
    from synth import edge_cases_city, edge_cases_vpq
    edge = json.load(open(os.path.join(G, "edge_cases.json")))
    for name, (pred, gt) in edge_cases_vpq().items():
        for a, b in zip(EO.vpq_stats(pred, gt), edge["vpq"][name]):
            assert a.tolist() == b, name
    for name, (pred, gt) in edge_cases_city().items():
        ev = EO.CityscapesPQOracle()
        ev.add_image(pred, gt)
        res, want = ev.evaluate(), edge["city"][name]
        assert (ev.TP, ev.FP, ev.FN, ev.iou_sum) == (want["tp"], want["fp"], want["fn"], want["iou_sum"]), name
        assert (res["pq"], res["sq"], res["rq"]) == (want["pq"], want["sq"], want["rq"]), name
        assert {str(c): {k: v for k, v in m.items()} for c, m in res["per_class"].items()} == want["per_class"], name
