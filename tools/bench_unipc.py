"""Sampling time and agreement of UniPC (orders 2 and 3) and DPM-Solver++ 2M against DDIM-50 at 5 to 10 UNet forwards,
on the flagship workload: sample() of 8 frames 384x1248 (latent 48x156) with the synthetic trained-like recipe of
bench.py (the same models, inputs, noise and fitted head, as tools/bench_dpm_solver.py).

Arms: DDIM-50 as the reference; DPM-Solver++ 2M, UniPC-2 and UniPC-3 (bh2, corrector at every step) at 5, 6, 8 and 10
forwards. Timing: CUDA events around each sample() call, after one untimed warm-up call of every arm; the arms
alternate inside every round (--rounds rounds), and the median over rounds is reported. Only the sampler loop is timed
(UNet forwards + scheduler updates). Agreement with DDIM-50: the merged panoptic ids and their categories pixel for
pixel, the relative L2 distance of the final latents, and PQ against the teacher ground truth made from the DDIM-50 ids
(bench.py's recipe). `fewest_forwards_matching_dpmpp2m10` names, per UniPC order, the fewest measured forwards whose ids
agree with DDIM-50 at least as well as DPM-Solver++ 2M at 10 forwards (null: none in the measured range). Everything
is reported, nothing asserted. The GPU name and power limit are read in the same run.

    python tools/bench_unipc.py [--rounds R] [--out FILE.json]
"""
import argparse
import copy
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from bench_dpm_solver import gpu_info  # noqa: E402
from video_latent_diffusion_panoptic_segmentation_b200 import _lib as L  # noqa: E402
from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.data import synthetic as SY  # noqa: E402
from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.evaluations import CityscapesPanopticEvaluator  # noqa: E402
from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.schedulers import (  # noqa: E402
    DDIMNoiseScheduler, DPMSolverMultistepScheduler, UniPCMultistepScheduler)
from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.trainers import TrainerDiffusion  # noqa: E402
from video_latent_diffusion_panoptic_segmentation_b200.tools import main_ldm  # noqa: E402

FORWARDS = (5, 6, 8, 10)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    L.lib()
    B, H, W = 8, 384, 1248
    h, w = H // 8, W // 8
    p = copy.deepcopy(main_ldm.BASE)
    vae, unet, ddim = main_ldm.build_models(p, dev, seed=0)
    tr = TrainerDiffusion(p=p, vae_semseg=vae, unet_model=unet, noise_scheduler=ddim, args={"gpu": 0})
    main_ldm.fit_trained_like_head(tr, (h, w), 50, seed=42, data_seed=1234)   # bench.py's head (DDIM-50 teacher)
    rgb = SY.trained_like_rgb_latents(B, h, w, seed=1234).to(dev)
    noise = torch.stack([torch.randn((4, h, w), generator=torch.Generator().manual_seed(42 + f)) for f in range(B)])
    noise = noise.to(dev)

    nk = p["noise_scheduler_kwargs"]
    sk = {k: nk[k] for k in ("num_train_timesteps", "beta_start", "beta_end", "beta_schedule")}
    s = DDIMNoiseScheduler(**nk, device=dev)
    s.set_timesteps_inference(50)
    s.move_timesteps_to(dev)
    arms = {"ddim50": (s, 50)}
    for n in FORWARDS:
        for name, s in ((f"dpmpp2m{n}", DPMSolverMultistepScheduler(**sk, solver_order=2)),
                        (f"unipc2_{n}", UniPCMultistepScheduler(**sk, solver_order=2)),
                        (f"unipc3_{n}", UniPCMultistepScheduler(**sk, solver_order=3))):
            s.set_timesteps(n, device=dev)
            arms[name] = (s, n)

    def run(name):
        s, n = arms[name]
        return tr.sample([""] * B, n, seed=None, rgb_latents=rgb, scheduler=s, noise=noise)

    latents = {name: run(name) for name in arms}           # warm-up of every arm (and the outputs compared below)
    torch.cuda.synchronize()
    times = {name: [] for name in arms}
    for r in range(args.rounds):
        order = list(arms) if r % 2 == 0 else list(arms)[::-1]
        for name in order:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            lat = run(name)
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1))
            assert torch.equal(lat, latents[name]), f"{name}: sample() is not deterministic"

    ref_lat = latents["ddim50"]
    _, ref_ids, _ = tr.panoptic_ids(ref_lat)
    ref_cat, _ = SY.split_cat_ins(ref_ids)
    gt = SY.teacher_ground_truth(ref_ids)
    t_ref = float(np.median(times["ddim50"]))
    res = {}
    for name, (s, n) in arms.items():
        _, ids, _ = tr.panoptic_ids(latents[name])
        cat, _ = SY.split_cat_ins(ids)
        ev = CityscapesPanopticEvaluator(device=dev)
        ev.add_images(ids, gt)
        pq = ev.evaluate()
        ms = float(np.median(times[name]))
        d = (latents[name] - ref_lat).pow(2).sum().sqrt() / ref_lat.pow(2).sum().sqrt()
        res[name] = {"unet_forwards": n, "ms_per_batch_median": round(ms, 2),
                     "ms_per_batch_all": [round(t, 2) for t in times[name]],
                     "speedup_vs_ddim50": round(t_ref / ms, 3),
                     "ids_agree_with_ddim50": round(float((ids == ref_ids).float().mean()), 5),
                     "category_agree_with_ddim50": round(float((cat == ref_cat).float().mean()), 5),
                     "latent_rel_l2_vs_ddim50": round(float(d), 5),
                     "pq_vs_ddim50_teacher_gt": round(float(pq["pq"]), 3)}
    target = res["dpmpp2m10"]["ids_agree_with_ddim50"]
    fewest = {f"unipc{q}": next((n for n in FORWARDS if res[f"unipc{q}_{n}"]["ids_agree_with_ddim50"] >= target), None)
              for q in (2, 3)}
    line = {"what": "sample() of one batch at 5-10 UNet forwards, UniPC (bh2) orders 2 / 3 vs DPM-Solver++ 2M, DDIM-50 "
                    "as the reference, trained-like synthetic recipe",
            "frames": B, "frame": [H, W], "latent": [h, w], "rounds": args.rounds, "gpu": gpu_info(0),
            "timing": "CUDA events around each sample() call (UNet forwards + updates), after one warm-up call per "
                      "arm; arms alternate within every round; median over rounds",
            "agreement": "against DDIM-50 on the same inputs and noise; pq_vs_ddim50_teacher_gt is PQ against a coarse, "
                         "partly relabelled copy of the DDIM-50 ids (bench.py's ground truth), so DDIM-50 itself scores "
                         "below 100",
            "dpmpp2m10_ids_agree_with_ddim50": target, "fewest_forwards_matching_dpmpp2m10": fewest,
            "arms": res}
    text = json.dumps(line)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
