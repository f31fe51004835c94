"""Streaming sampler (TrainerDiffusion.sample_stream) against the batch sampler, on 64 frames of 384x1248 (latent
48x156) at B = 8 with the trained-like synthetic models of bench.py, for DPM-Solver++ 2M-10, UniPC-2-8 and DDIM-50.

Two arrival patterns:
  all_at_once  every frame is available at t = 0. Stream: sample_stream over the 64 frames. Batch: sample() on 8
               batches of 8, one after the other.
  fixed_rate   frame f arrives at f * period. Stream: sample_stream, fed each frame once it has arrived. Batch: sample()
               at B = 1 on each frame once it has arrived and the previous one is done. The period is
               --load_factor (default 1.5) times the stream's per-frame time of the all_at_once pattern, so the stream
               runs at 1 / load_factor of its capacity.
Reported per arm: frames/s (frames over first arrival to last finish) and per-frame latency, median and p95, from
arrival and from admission (a stream frame entering a slot; a batch frame's sample() call starting) to the frame's
latents being final on the device (a CUDA event recorded when the frame is handed out, converted to the host clock
through a reference event). Every stream frame's latents are also checked against the batch path's bit for bit where
the batch path runs it in a batch of the same size at the same position (all_at_once). The GPU name and power limit
are read in the same run.

    python tools/bench_stream.py [--frames 64] [--load_factor 1.5] [--out FILE.json]
"""
import argparse
import copy
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from bench_dpm_solver import gpu_info  # noqa: E402
from video_latent_diffusion_panoptic_segmentation_b200 import _lib as L  # noqa: E402
from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.data import synthetic as SY  # noqa: E402
from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.schedulers import (  # noqa: E402
    DDIMNoiseScheduler, DPMSolverMultistepScheduler, UniPCMultistepScheduler)
from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.trainers import TrainerDiffusion  # noqa: E402
from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.trainers.trainers_ldm_cond import stream_noise  # noqa: E402
from video_latent_diffusion_panoptic_segmentation_b200.tools import main_ldm  # noqa: E402

B, SEED = 8, 42


class Clock:
    """Host clock with a device reference: event times map onto perf_counter seconds."""

    def __init__(self):
        torch.cuda.synchronize()
        self.ref = torch.cuda.Event(enable_timing=True)
        self.ref.record()
        torch.cuda.synchronize()
        self.t0 = time.perf_counter()

    def now(self):
        return time.perf_counter() - self.t0

    def mark(self):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    def at(self, event):
        return self.ref.elapsed_time(event) / 1e3


def summary(arrive, admit, finish):
    n = len(finish)
    fin = np.array([finish[f] for f in range(n)])
    lat_arr = fin - np.array([arrive[f] for f in range(n)])
    lat_adm = fin - np.array([admit[f] for f in range(n)])
    span = fin.max() - min(arrive.values())
    return {"frames_per_s": round(n / span, 3),
            "latency_ms_from_arrival": {"median": round(1e3 * float(np.median(lat_arr)), 1),
                                        "p95": round(1e3 * float(np.percentile(lat_arr, 95)), 1)},
            "latency_ms_from_admission": {"median": round(1e3 * float(np.median(lat_adm)), 1),
                                          "p95": round(1e3 * float(np.percentile(lat_adm, 95)), 1)}}


def run_stream(tr, sched, N, rgb, period):
    """sample_stream over all frames; frame f becomes available at f * period (0: all at once)."""
    n = rgb.shape[0]
    clk = Clock()
    arrive = {f: f * period for f in range(n)}
    admit, finish_ev, out = {}, {}, {}

    def frames():
        f = 0
        while f < n:
            if clk.now() < arrive[f]:
                if len(admit) > len(out):
                    yield None        # frames in flight: the next forward runs without this one
                    continue
                time.sleep(max(0.0, arrive[f] - clk.now()))   # every slot empty: wait for the frame
            admit[f] = clk.now()
            yield f, rgb[f:f + 1], None
            f += 1

    for fid, lat in tr.sample_stream(frames(), N, scheduler=sched, batch_size=B, seed=SEED):
        finish_ev[fid] = clk.mark()
        out[fid] = lat
    torch.cuda.synchronize()
    return summary(arrive, admit, {f: clk.at(e) for f, e in finish_ev.items()}), out


def run_batch(tr, sched, N, rgb, period, bsz):
    """sample() on consecutive batches of bsz frames; a batch starts once its last frame has arrived and the previous
    batch is done."""
    n = rgb.shape[0]
    h, w = rgb.shape[-2:]
    clk = Clock()
    arrive = {f: f * period for f in range(n)}
    admit, finish_ev, out = {}, {}, {}
    for k in range(0, n, bsz):
        fs = list(range(k, min(k + bsz, n)))
        while clk.now() < arrive[fs[-1]]:
            time.sleep(min(1e-4, arrive[fs[-1]] - clk.now()))
        noise = torch.cat([stream_noise(f, SEED, (4, h, w)) for f in fs])
        for f in fs:
            admit[f] = clk.now()
        lat = tr.sample([""] * len(fs), N, rgb_latents=rgb[k:k + len(fs)], scheduler=sched, noise=noise)
        e = clk.mark()
        torch.cuda.synchronize()        # the next batch starts after this one, as a caller of sample() would see it
        for i, f in enumerate(fs):
            finish_ev[f], out[f] = e, lat[i:i + 1]
    return summary(arrive, admit, {f: clk.at(e) for f, e in finish_ev.items()}), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=64)
    ap.add_argument("--load_factor", type=float, default=1.5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    L.lib()
    H, W = 384, 1248
    h, w = H // 8, W // 8
    p = copy.deepcopy(main_ldm.BASE)
    vae, unet, _ = main_ldm.build_models(p, dev, seed=0)
    tr = TrainerDiffusion(p=p, vae_semseg=vae, unet_model=unet, args={"gpu": 0})
    rgb = SY.trained_like_rgb_latents(args.frames, h, w, seed=1234).to(dev)

    nk = p["noise_scheduler_kwargs"]
    sk = {k: nk[k] for k in ("num_train_timesteps", "beta_start", "beta_end", "beta_schedule")}
    arms = {}
    s = DDIMNoiseScheduler(**nk, device=dev)
    s.set_timesteps_inference(50)
    arms["ddim50"] = (s, 50)
    s = DPMSolverMultistepScheduler(**sk, solver_order=2)
    s.set_timesteps(10, device=dev)
    arms["dpmpp2m10"] = (s, 10)
    s = UniPCMultistepScheduler(**sk, solver_order=2)
    s.set_timesteps(8, device=dev)
    arms["unipc2_8"] = (s, 8)

    res = {}
    for name, (s, N) in arms.items():
        # warm-up: every plan and graph of this arm (stream B, batch B and B = 1) is built outside the timed runs
        run_stream(tr, s, N, rgb[:B + 1], 0.0)
        run_batch(tr, s, N, rgb[:B + 1], 0.0, B)
        run_batch(tr, s, N, rgb[:1], 0.0, 1)
        a_stream, out_s = run_stream(tr, s, N, rgb, 0.0)
        a_batch, out_b = run_batch(tr, s, N, rgb, 0.0, B)
        same = all(torch.equal(out_s[f], out_b[f]) for f in range(args.frames))
        period = args.load_factor * (args.frames / a_stream["frames_per_s"]) / args.frames
        f_stream, _ = run_stream(tr, s, N, rgb, period)
        f_b1, _ = run_batch(tr, s, N, rgb, period, 1)
        res[name] = {"unet_forwards": N,
                     "all_at_once": {"stream_B8": a_stream, "sample_batches_of_8": a_batch,
                                     "stream_latents_equal_batch_bit_for_bit": same},
                     "fixed_rate": {"arrival_period_ms": round(1e3 * period, 2),
                                    "arrivals_per_s": round(1 / period, 3),
                                    "stream_B8": f_stream, "sample_B1_per_frame": f_b1}}
        print(json.dumps({name: res[name]}), flush=True)
    line = {"what": "sample_stream at B = 8 against sample() (batches of 8 with all frames available; B = 1 per frame "
                    "with frames arriving at a fixed rate), trained-like synthetic recipe",
            "frames": args.frames, "frame": [H, W], "latent": [h, w], "slots": B, "load_factor": args.load_factor,
            "gpu": gpu_info(0),
            "timing": "host clock for arrivals and admissions; a CUDA event per finished frame, mapped onto the host "
                      "clock through a reference event; every plan built in an untimed warm-up run",
            "arms": res}
    text = json.dumps(line)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
