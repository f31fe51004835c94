#!/usr/bin/env python
"""Benchmark of the LDMSeg sampler hot path (BASELINE.json metric: panoptic frames/sec, DDIM-50, 384x1248 KITTI).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config NAME[,NAME...]]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Workloads (`--config`, one JSON line each; the default is the one BASELINE.json's metric is quoted on):
  batch8        configs[1]: 8 frames 384x1248 per GPU, DDIM 50 (weak scaling: the clip is all ranks' frames)
  clip8_strong  configs[2]: ONE 8-frame clip, frames split 8/N per GPU, DVPQ windows of 1 and 2 frames (strong scaling)
  seq1101       configs[3]: a 1101-frame sequence sharded contiguously over the ranks, batches of 8, DVPQ k = 1 and 2
  k2            configs[4]: 768x2496 frames (latent 96x312), 2 frames per GPU, DDIM 50 (weak scaling)
One "step" = one pass of the hot path over this rank's frames of the clip: per batch  noise -> T x (UNet, DDIM update)
-> seg-AE decode -> fused argmax/threshold ids -> merge -> PQ statistics;  then the PQ reduction and the DVPQ statistics
over the whole clip (halo all_gather + stats all_reduce at N > 1). Weights: random init + the "trained-like" recipe
(ldmseg/models/unet_init.py), so the predictions are not degenerate; ground truth: a coarse, partly mislabelled copy
of a teacher pass of the same pipeline (ldmseg/data/synthetic.py). Rank 0 prints ONE JSON line per config (DESIGN.md
"Measurement" explains every field).
"""
import argparse
import copy
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "panoptic frames/sec (DDIM-50, 384x1248 KITTI)"
# analytic work model of BASELINE.md section 3, per frame
WORK = {(384, 1248): {"unet_step": 1597.2e9, "ae": 90.4e9}, (768, 2496): {"unet_step": 11294.0e9, "ae": 361.7e9}}
CONFIGS = {
    "batch8": dict(frame=(384, 1248), frames_per_gpu=8, batch=8, scaling="weak", dvpq_k=(2,), baseline="configs[1]"),
    "clip8_strong": dict(frame=(384, 1248), clip_frames=8, batch=8, scaling="strong", dvpq_k=(1, 2), baseline="configs[2]"),
    "seq1101": dict(frame=(384, 1248), clip_frames=1101, batch=8, scaling="strong", dvpq_k=(1, 2), baseline="configs[3]"),
    "k2": dict(frame=(768, 2496), frames_per_gpu=2, batch=2, scaling="weak", dvpq_k=(2,), baseline="configs[4]"),
}


def workload_text(name, cfg, n_frames, ddim_steps, world):
    H, W = cfg["frame"]
    what = {"batch8": f"batch {cfg.get('frames_per_gpu')} frames {H}x{W} per GPU",
            "clip8_strong": f"one {n_frames}-frame clip of {H}x{W} frames split over the GPUs",
            "seq1101": f"a {n_frames}-frame sequence of {H}x{W} frames (SemanticKITTI-shaped, 376x1241 padded) sharded "
                       f"contiguously over the GPUs, batches of {cfg['batch']}",
            "k2": f"batch {cfg.get('frames_per_gpu')} frames {H}x{W} per GPU (latent {H // 8}x{W // 8})"}[name]
    return (f"LDMSeg sampler, {what}, DDIM {ddim_steps} steps, random-init UNet (815M, SD-1.4 topology, self-attn only) "
            f"+ seg-AE with the trained-like recipe, bf16 storage / fp32 accumulate, incl. AE decode, ids, merge, PQ "
            f"stats and DVPQ stats (windows of {'/'.join(str(k) for k in cfg['dvpq_k'])} frames over the clip formed by "
            f"all ranks' frames: halo all_gather + stats all_reduce)")


def config_dict(name, cfg, n_frames, ddim_steps, world):
    return {"workload": workload_text(name, cfg, n_frames, ddim_steps, world), "name": name,
            "baseline_config": cfg["baseline"], "clip_frames": n_frames, "frame": list(cfg["frame"]),
            "frames_per_gpu": (n_frames + world - 1) // world, "batch": cfg["batch"], "ddim_steps": ddim_steps,
            "parallelism": f"frames sharded contiguously over {world} GPU(s)",
            "l2": "per-step working set (weights 1.6 GB + activations) exceeds the 126 MB L2"}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return d["hbm_gbs"], d["bf16_tflops"], d.get("bf16_tflops_sustained", d["bf16_tflops"]), "measured"
    return 6650.0, 1590.0, 1400.0, "fallback"  # B200_PROFILING.md fallback


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        self.gpu, self.lines, self.proc = gpu, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------- reference arm
class CpuReference:
    """The reference's CPU path for this metric, bounded: the oracle (reference scheduler / seg-AE decoder / merge /
    evaluator restated and pinned by tests/golden; UNet = restated diffusers, which is not installable here) on ONE
    frame. One `unet_step()` = one DDIM iteration (UNet fp32 + scheduler step); `tail()` = seg-AE decode + ids/merge +
    PQ + one DVPQ window. frames/s is extrapolated to `ddim_steps` iterations."""

    def __init__(self, ddim_steps, frame=(384, 1248), threads=None):
        from oracle import ldmseg_oracle as LO
        from oracle import unet_oracle as UO
        from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.data import trained_like_rgb_latents
        from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.models import unet_init
        self.LO = LO
        self.threads = threads or os.cpu_count()
        torch.set_num_threads(self.threads)
        self.T, self.frame = ddim_steps, frame
        h, w = frame[0] // 8, frame[1] // 8
        self.unet = UO.build_unet(seed=0, model_kwargs=unet_init.TRAINED_LIKE_MODEL_KWARGS)
        self.unet.load_state_dict(unet_init.trained_like_unet_(dict(self.unet.state_dict())))
        self.vae = LO.build_seg_decoder(seed=1)
        self.vae.load_state_dict(unet_init.trained_like_seg_decoder_(dict(self.vae.state_dict())))
        self.sched = LO.DDIMOracle()
        self.sched.set_timesteps_inference(ddim_steps)
        self.rgb = trained_like_rgb_latents(1, h, w)
        self.lat = torch.randn((1, 4, h, w), generator=torch.Generator().manual_seed(42))
        self.gt = np.random.default_rng(7).integers(0, 19, size=frame).astype(np.int64)
        self.i = 0

    def unet_step(self):
        t = self.sched.timesteps[self.i % len(self.sched.timesteps)]
        self.i += 1
        t0 = time.perf_counter()
        with torch.no_grad():
            eps = self.unet(torch.cat([self.lat, self.rgb], 1), t, encoder_hidden_states=None)
            self.lat, _ = self.sched.step(eps, t, self.lat)
        return time.perf_counter() - t0

    def tail(self):
        from oracle import eval_oracle as EO
        t0 = time.perf_counter()
        with torch.no_grad():
            logits = self.LO.decode_latents(self.vae, self.lat)
            _, cleaned, _ = self.LO.logits_to_panoptic(logits[0], 0.5, 512, 0.5, 127)
        ev = EO.CityscapesPQOracle()
        ev.add_image(cleaned, self.gt)
        # one DVPQ window of 2 frames per frame, as in our arm (the clip's frames are this frame repeated)
        void = cleaned < 0
        pc = np.where(void, 19, cleaned % 19).astype(np.int32)
        pi = np.where(void, 0, cleaned // 19).astype(np.int32)
        gc, gi = self.gt.astype(np.int32), np.zeros_like(self.gt, dtype=np.int32)
        EO.dvpq_window([pc, pc], [pi, pi], [gc, gc], [gi, gi])
        return time.perf_counter() - t0

    def describe(self, t_unet, t_tail, n):
        H, W = self.frame
        return (f"BOUNDED SAMPLE, extrapolated: 1 frame {H}x{W} on {self.threads} host threads, {n} of {self.T} DDIM "
                f"iterations timed (UNet fp32 + scheduler, {t_unet:.2f} s each) + seg-AE decode + ids/merge + PQ + one "
                f"DVPQ window ({t_tail:.2f} s); frames/s = 1 / ({self.T} x iteration + tail). fp32 CPU port of the "
                f"reference path (the reference's diffusers UNet is not installable here, the oracle restatement stands in)")


def cpu_reference_sample(ddim_steps, frame, unet_iters=3):
    ref = CpuReference(ddim_steps, frame)
    ref.unet_step()  # untimed warm-up (thread pool, allocator)
    t_unet = float(np.mean([ref.unet_step() for _ in range(unet_iters)]))
    t_tail = ref.tail()
    return {"fps": 1.0 / (ddim_steps * t_unet + t_tail), "cores": ref.threads,
            "sample": ref.describe(t_unet, t_tail, unet_iters)}


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    name = args.config.split(",")[0]
    cfg = CONFIGS[name]
    world = args.gpus
    n_frames = cfg.get("clip_frames") or cfg["frames_per_gpu"] * world
    ref = CpuReference(args.ddim_steps, cfg["frame"])
    t_tail = ref.tail()
    for _ in range(args.warmup):
        ref.unet_step()
    times = [ref.unet_step() for _ in range(args.steps)]
    t_unet = float(np.mean(times))
    fps = 1.0 / (args.ddim_steps * t_unet + t_tail)
    cd = config_dict(name, cfg, n_frames, args.ddim_steps, world)
    cd["reference_arm"] = ("bounded sample of this workload: ONE frame, `steps` = DDIM iterations of that frame (not "
                           "batches), frames/s extrapolated to the full DDIM schedule; see cpu_baseline.sample")
    line = {"impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
            "steps": len(times), "warmup": args.warmup, "ms_per_step": 1e3 * t_unet, "higher_is_better": True,
            "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cd,
            "step_is": "one DDIM iteration (UNet fp32 + scheduler step) of ONE frame; extrapolated=true",
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": ref.threads, "kind": "port",
                             "sample": ref.describe(t_unet, t_tail, len(times))},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# ------------------------------------------------------------------------------------------------- our arm
def frame_digests(ids):
    """[n, H, W] int32 device tensor -> list of per-frame sha256 prefixes."""
    a = np.ascontiguousarray(ids.detach().to("cpu", torch.int32).numpy())
    return [hashlib.sha256(a[i].tobytes()).hexdigest()[:12] for i in range(a.shape[0])]


DUMP_BYTES = 64 * 10 ** 6   # --dump-outputs writes at most this much, split evenly over the configs of the run
PQ_FIELDS = ("pq", "sq", "rq", "tp", "fp", "fn", "iou_sum", "thing_pq", "thing_sq", "thing_rq", "stuff_pq", "stuff_sq",
             "stuff_rq")
CLASS_FIELDS = ("pq", "sq", "rq", "tp", "fp", "fn")
DVPQ_FIELDS = ("iou", "tp", "fn", "fp")


def dump_outputs(out_dir, name, wl, res, budget):
    """What the last timed step returned to its caller, one float array per file out_dir/<config>_<array>.npy:
      ids            merged panoptic ids (-1 = void) of rank 0's frames, float32 [frames, H, W]; when all frames would
                     exceed `budget` bytes, a fixed seeded sample of whole frames
      ids_frames     global index of each frame in `ids`, float64
      pq             the PQ evaluator's totals in PQ_FIELDS order, float64
      pq_per_class   one row per class present: class id, then CLASS_FIELDS, float64
      dvpq_k<k>      DVPQ statistics over windows of k frames, rows DVPQ_FIELDS x 19 classes, float64
      dvpq_k<k>_pq   pq, pq_things, pq_stuff, number of windows, float64
    PQ and DVPQ cover the whole clip (all ranks)."""
    os.makedirs(out_dir, exist_ok=True)
    frame_bytes = wl.H * wl.W * 4
    keep = np.arange(wl.n_local)
    if wl.n_local * frame_bytes > budget:
        keep = np.sort(np.random.default_rng(0).choice(wl.n_local, max(1, budget // frame_bytes), replace=False))
    arrays = {
        "ids": wl.ids_host.numpy()[keep].astype(np.float32),   # ids are below 2^24: exact in float32
        "ids_frames": (wl.lo + keep).astype(np.float64),
        "pq": np.array([res[k] for k in PQ_FIELDS], np.float64),
        "pq_per_class": np.array([[c] + [m[k] for k in CLASS_FIELDS] for c, m in sorted(res["per_class"].items())],
                                 np.float64).reshape(-1, 1 + len(CLASS_FIELDS)),
    }
    for k, v in res["dvpq"].items():
        arrays[f"dvpq_k{k}"] = np.stack([np.asarray(v[f], np.float64) for f in DVPQ_FIELDS])
        arrays[f"dvpq_k{k}_pq"] = np.array([v["pq"], v["pq_things"], v["pq_stuff"], v["n_windows"]], np.float64)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}_{k}.npy"), a)


class Workload:
    """This rank's contiguous share [lo, hi) of an n_frames clip, its synthetic inputs, and one pass over it."""

    def __init__(self, name, args, env):
        from video_latent_diffusion_panoptic_segmentation_b200.eval import clip_dvpq as CD
        from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.data import synthetic as SY
        from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.evaluations import CityscapesPanopticEvaluator
        from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.trainers import TrainerDiffusion
        from video_latent_diffusion_panoptic_segmentation_b200.tools import main_ldm
        self.name, self.cfg, self.env, self.args = name, CONFIGS[name], env, args
        self.CD, self.SY = CD, SY
        cfg, world, rank, dev = self.cfg, env["world"], env["rank"], env["dev"]
        self.T = args.ddim_steps
        self.H, self.W = cfg["frame"]
        self.h, self.w = self.H // 8, self.W // 8
        fpg = args.frames_per_gpu or cfg.get("frames_per_gpu")
        self.n_frames = args.clip_frames or cfg.get("clip_frames") or fpg * world
        self.lo, self.hi = CD.shard_range(self.n_frames, rank, world)
        self.n_local = self.hi - self.lo
        self.batch = min(cfg["batch"], max(1, self.n_local))
        p = copy.deepcopy(main_ldm.BASE)
        p["sampling_kwargs"]["num_inference_steps"] = self.T
        self.vae, self.unet, self.sched = env["models"]
        self.tr = TrainerDiffusion(p=p, vae_semseg=self.vae, unet_model=self.unet, noise_scheduler=self.sched,
                                   args={"gpu": env["local"]})
        self.sched.set_timesteps_inference(self.T)
        self.sched.move_timesteps_to(dev)
        # step 4 of the recipe: the head is fitted to a batch-1 teacher sample of global frame 0 at this frame size
        # (the same on every rank and at every world size)
        main_ldm.fit_trained_like_head(self.tr, (self.h, self.w), self.T, seed=42, data_seed=1234)
        self.evaluator = CityscapesPanopticEvaluator(device=dev)
        # synthetic inputs of the local frames: pinned host copies (e2e arm) + device-resident copies (`value`)
        n = self.n_local
        self.rgb_host = SY.trained_like_rgb_latents(n, self.h, self.w, seed=1234, first_frame=self.lo).pin_memory()
        self.rgb_dev = self.rgb_host.to(dev)
        # Noise belongs to the GLOBAL frame (seed 42 + frame index), so a frame gets the same noise whatever the world
        # size and batch split are -- the ids digests of different N are then comparable. (The reference re-seeds one
        # generator per batch, :1091-1095, :1246: its noise depends on how the sampler happened to batch the frames.)
        self.noise_host = torch.stack([torch.randn((4, self.h, self.w), generator=torch.Generator().manual_seed(42 + f))
                                       for f in range(self.lo, self.hi)]).pin_memory() if n else torch.empty((0, 4, self.h, self.w))
        self.noise_dev = self.noise_host.to(dev)
        self.ids_host = torch.empty((n, self.H, self.W), dtype=torch.int32).pin_memory()
        self.cleaned = torch.empty((n, self.H, self.W), dtype=torch.int32, device=dev)
        self.gt_dev = torch.zeros((n, self.H, self.W), dtype=torch.int32, device=dev)
        self.gt_host = None

    def batches(self):
        for a in range(0, self.n_local, self.batch):
            yield a, min(a + self.batch, self.n_local)

    def make_ground_truth(self):
        """Teacher pass (also the first warm-up): GT = coarse, partly mislabelled copy of this pipeline's own prediction."""
        for a, b in self.batches():
            lat = self.tr.sample([""] * (b - a), self.T, seed=None, rgb_latents=self.rgb_dev[a:b], scheduler=self.sched,
                                 noise=self.noise_dev[a:b])
            _, cleaned, _ = self.tr.panoptic_ids(lat)
            self.gt_dev[a:b] = self.SY.teacher_ground_truth(cleaned)
        self.gt_host = self.gt_dev.cpu().pin_memory()
        self.gt_cat, self.gt_ins = self.SY.split_cat_ins(self.gt_dev, ignore=0)

    def step(self, resident):
        from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.trainers.trainers_ldm_cond import reduce_evaluator_
        dev, world = self.env["dev"], self.env["world"]
        self.evaluator.reset()
        for a, b in self.batches():
            if resident:
                rgb, noise, gt = self.rgb_dev[a:b], self.noise_dev[a:b], self.gt_dev[a:b]
            else:   # host buffers in, ids out: the copies are part of the timed region
                rgb = self.rgb_host[a:b].to(dev, non_blocking=True)
                noise = self.noise_host[a:b]
                gt = self.gt_host[a:b].to(dev, non_blocking=True)
            lat = self.tr.sample([""] * (b - a), self.T, seed=None, rgb_latents=rgb, scheduler=self.sched, noise=noise)
            _, cleaned, _ = self.tr.panoptic_ids(lat)
            self.cleaned[a:b] = cleaned
            self.evaluator.add_images(cleaned, gt)    # one labelling + one histogram launch + one D2H per batch
            if not resident:
                self.ids_host[a:b].copy_(cleaned, non_blocking=True)   # the panoptic ids a caller reads back
        if world > 1:
            reduce_evaluator_(self.evaluator, dev)
        res = self.evaluator.evaluate()
        pc, pi = self.SY.split_cat_ins(self.cleaned)
        res["dvpq"] = {k: self.CD.dvpq_clip_sharded(pc, pi, self.gt_cat, self.gt_ins, n_frames=self.n_frames,
                                                    eval_frames=k) for k in self.cfg["dvpq_k"] if self.n_frames >= k}
        if not resident:
            torch.cuda.current_stream().synchronize()
        return res

    def h2d_d2h_bytes(self):
        n = self.n_local
        per_frame_in = 4 * self.h * self.w * 4 * 2 + self.H * self.W * 4     # rgb latents + noise + ground truth
        return int(n * per_frame_in), int(n * self.H * self.W * 4)


def run_config(name, args, env):
    import torch.distributed as dist
    from video_latent_diffusion_panoptic_segmentation_b200 import _lib as L
    from video_latent_diffusion_panoptic_segmentation_b200 import ops
    world, rank, local, dev = env["world"], env["rank"], env["local"], env["dev"]
    wl = Workload(name, args, env)
    cfg, T, B = wl.cfg, wl.T, wl.batch
    wl.make_ground_truth()

    def timed(resident, warmup, steps, sample_clocks=False):
        for _ in range(warmup):
            wl.step(resident)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        cs = ClockSampler(local) if sample_clocks else None
        if cs:
            cs.start()
        try:
            n0 = L.launch_count()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                res = wl.step(resident)
            e1.record()
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            ms = e0.elapsed_time(e1)
        finally:   # the sampler is a child process: never leave it running
            clocks = cs.stop() if cs else None
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, res, L.launch_count() - n0, clocks

    # a long sequence is its own warm-up: W counts passes for the short clips, and at most one pass for seq1101
    warm = args.warmup if wl.n_local <= 16 else min(args.warmup, 1)
    ms, res, eager_launches, clocks = timed(True, warm, args.steps, sample_clocks=True)
    plan = wl.tr._loop_state(B, wl.h, wl.w)["plan"]
    n_batches = len(list(wl.batches()))
    graph_launches = plan.launches_per_forward * T * n_batches * args.steps if plan.graph is not None else 0
    fps = wl.n_frames * args.steps / (ms / 1e3)
    ms_e2e, res_e2e, _, _ = timed(False, 1 if warm else 0, args.steps)      # same number of steps as `value`
    fps_e2e = wl.n_frames * args.steps / (ms_e2e / 1e3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, name, wl, res_e2e, DUMP_BYTES // len(args.config.split(",")))

    # digests: identical ids / integer statistics at N = 1 and N > 1 for the same global frames
    digs = frame_digests(wl.cleaned)
    if world > 1:
        allp = [None] * world
        dist.all_gather_object(allp, (wl.lo, digs))
        digs = [d for _, ds in sorted(allp) for d in ds]
    h2d, d2h = wl.h2d_d2h_bytes()
    hbm, tf_burst, tf_sus, which = peaks()
    work = WORK[tuple(cfg["frame"])]
    dv = res["dvpq"]
    line = {"metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": warm, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": cfg["scaling"],
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": config_dict(name, cfg, wl.n_frames, T, world),
            "e2e": {"value": fps_e2e, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": args.steps},
            "gpu_launches": int(graph_launches + eager_launches),
            "clocks": clocks, "pq": {k: res[k] for k in ("pq", "sq", "rq", "tp", "fp", "fn")},
            "dvpq": {f"k{k}": {"pq": float(v["pq"]), "windows": int(v["n_windows"]), "tp": int(v["tp"].sum()),
                               "fn": int(v["fn"].sum()), "fp": int(v["fp"].sum())} for k, v in dv.items()},
            "ids_digest": {"frames": len(digs), "per_frame_first16": digs[:16],
                           "all": hashlib.sha256("".join(digs).encode()).hexdigest()[:16],
                           "first8": hashlib.sha256("".join(digs[:8]).encode()).hexdigest()[:16],
                           "note": "sha256 of the merged int32 id map of every global frame, in frame order (noise and "
                                   "inputs belong to the global frame). `first8` covers global frames 0-7: in the weak-"
                                   "scaling configs it is the same at every N (same frames, same batch of 8 per GPU = "
                                   "the same kernels: bit-identical ids). In the strong-scaling configs the batch per GPU "
                                   "changes with N, and with it the tiling (block_n, split-K, GroupNorm slices) and the "
                                   "fp32 summation order: ids then agree up to bf16 rounding flips, see pq / dvpq"},
            # nominal FLOPs of the reference's operators per frame (SURVEY 8d); roofline.achieved counts EXECUTED ones
            "whole_job_frac_of_tensor_peak": fps / world * (T * work["unet_step"] + work["ae"]) / (tf_sus * 1e12)}

    if rank == 0:
        extras(line, wl, plan, args, env)
        emit(line)
    del wl
    torch.cuda.empty_cache()


def extras(line, wl, plan, args, env):
    """Rank 0, outside the timed region: roofline of the dominant kernel, phase split, HBM kernels, baselines."""
    from video_latent_diffusion_panoptic_segmentation_b200 import ops
    dev, world = env["dev"], env["world"]
    T, B, name = wl.T, wl.batch, wl.name
    hbm, tf_burst, tf_sus, which = peaks()

    def phases():
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        a, b = next(wl.batches())
        wl.evaluator.reset()
        ev[0].record()
        lat = wl.tr.sample([""] * (b - a), T, seed=None, rgb_latents=wl.rgb_dev[a:b], scheduler=wl.sched,
                           noise=wl.noise_dev[a:b])
        ev[1].record()
        _, cleaned, _ = wl.tr.panoptic_ids(lat)
        ev[2].record()
        wl.evaluator.add_images(cleaned, wl.gt_dev[a:b])
        wl.evaluator.evaluate()
        ev[3].record()
        pc, pi = wl.SY.split_cat_ins(cleaned)
        if world == 1:
            wl.CD.dvpq_clip_sharded(pc, pi, wl.gt_cat[a:b], wl.gt_ins[a:b], n_frames=b - a, eval_frames=min(2, b - a))
        ev[4].record()
        torch.cuda.synchronize()
        return {"sampler_unet_ddim": ev[0].elapsed_time(ev[1]), "ae_decode_ids_merge": ev[1].elapsed_time(ev[2]),
                "pq_evaluator": ev[2].elapsed_time(ev[3]), "dvpq_k2_one_batch": ev[3].elapsed_time(ev[4])}

    line["phases_ms_per_batch"] = {k: round(v, 2) for k, v in phases().items()}

    # roofline of the dominant kernel (gemm_tc_kernel: linear / conv1x1 / implicit conv3x3), measured live with
    # CUDA events around every launch of one eager UNet forward
    prof = wl.unet.profile_plan(plan, iters=2)
    if args.profile_out:
        with open(args.profile_out, "w") as f:
            json.dump(prof, f, default=str)
    by = {}
    for r in prof:
        d = by.setdefault(r["op"], {"ms": 0.0, "flops": 0, "n": 0})
        d["ms"] += r["ms"]; d["flops"] += r["flops"]; d["n"] += 1
    tot_ms = sum(d["ms"] for d in by.values())
    gm = by.get("gemm", {"ms": 1e-9, "flops": 0, "n": 1})
    ach = gm["flops"] / (gm["ms"] / 1e3) / 1e12
    traffic, traffic_src = None, None
    import glob
    tpaths = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_unet_forward_traffic.json")))
    if tpaths and name == "batch8":
        tj = json.load(open(tpaths[-1]))
        if "gemm_tc_kernel" in tj:
            traffic = tj["gemm_tc_kernel"]["dram_bytes_per_launch"]
            traffic_src = f"not measured in this run: from the committed ncu capture profiles/{os.path.basename(tpaths[-1])}"
    line["roofline"] = {"bound": "tensor", "kernel": "gemm_tc_kernel", "achieved": ach, "peak": tf_sus,
                        "unit": "TFLOP/s", "frac": ach / tf_sus, "peak_source": f"{which} (sustained bf16)",
                        "traffic": traffic, "traffic_source": traffic_src, "launches": gm["n"],
                        "avg_launch_us": gm["ms"] * 1e3 / max(1, gm["n"]),
                        "share_of_unet_step": gm["ms"] / tot_ms}
    line["breakdown_ms_per_unet_forward"] = {k: round(v["ms"], 3) for k, v in sorted(by.items(), key=lambda kv: -kv[1]["ms"])}
    at = by.get("flash_attn")
    if at:
        line["attention_tflops"] = at["flops"] / (at["ms"] / 1e3) / 1e12
    hb = {"bytes": 0, "ms": 0.0}
    for r in prof:
        # the first-level launches only (>= 38 MB): the small levels are launch-latency bound in this eager profile
        if r["op"] in ("groupnorm", "layernorm") and r["bytes"] >= 38e6:
            hb["bytes"] += r["bytes"] * 2 // 3 if r["op"] == "groupnorm" else r["bytes"]  # 1R + 1W (see DESIGN.md)
            hb["ms"] += r["ms"]
    if hb["ms"] > 0:
        gbs = hb["bytes"] / (hb["ms"] / 1e3) / 1e9
        line["hbm_kernels"] = {"kernels": "gn_fused, layernorm_rows", "achieved": gbs, "peak": hbm, "unit": "GB/s",
                               "frac": gbs / hbm, "note": "first-level launches (>= 38 MB), CUDA events around each launch"}
    if name != "batch8":
        return

    def hbm_tail_kernels():
        """The integer kernels that are pure streaming (north_star: >= 70 % of HBM peak on the elementwise / scheduler /
        bit-decode kernels), each timed alone with CUDA events at the full frame size; inputs larger than L2."""
        out = {}
        H, W = wl.H, wl.W
        bits = torch.randn((8, 16, H, W), device=dev)                    # 16 bit planes of 8 frames: 245 MB
        ids = torch.empty((8, H, W), dtype=torch.int32, device=dev)
        planes = torch.empty((8, 16, H, W), dtype=torch.float32, device=dev)
        cases = {
            "decode_bitmap16": (lambda: ops.decode_bitmap(bits, ids), bits.numel() * 4 + ids.numel() * 4),
            "encode_bitmap16": (lambda: ops.encode_bitmap(ids, planes, 255, 0.5), planes.numel() * 4 + ids.numel() * 4),
        }
        ids.random_(0, 128)
        for nm, (fn, nbytes) in cases.items():
            for _ in range(3):
                fn()
            a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(10):
                fn()
            b_.record()
            torch.cuda.synchronize()
            us = a.elapsed_time(b_) * 100.0
            out[nm] = {"us": round(us, 2), "gbs": round(nbytes / us / 1e3, 1), "bytes": int(nbytes),
                       "frac": round(nbytes / us / 1e3 / hbm, 3)}
        out["peak_gbs"] = hbm
        return out

    def rgb_vae_encode_ms():
        """The step in front of the metric's timed region (SURVEY 8f rank 1, excluded from the metric by 8d): 8 frames
        through the RGB VAE encoder (random-init SD-1.4 VAE), CUDA events, reported for context only."""
        from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.models import GeneralVAEImage, unet_init
        vim = GeneralVAEImage.from_pretrained(state_dict=unet_init.random_vae_image_state_dict(seed=2), device=dev)
        img = torch.rand((8, 3, wl.H, wl.W), device=dev)
        for _ in range(2):
            vim.encode_moments(img, scale=2.0, shift=-1.0)
        a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(3):
            vim.encode_moments(img, scale=2.0, shift=-1.0)
        b_.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b_) / 3

    for key, fn in (("hbm_tail_kernels", hbm_tail_kernels), ("rgb_vae_encode_ms_per_batch", rgb_vae_encode_ms)):
        try:
            line[key] = fn()
        except Exception as e:  # context only: never take the measurement down
            line[key] = f"failed: {e!r}"
        torch.cuda.empty_cache()
    if world == 1 and not args.no_gpu_baseline:
        try:
            line["torch_gpu_baseline"] = torch_gpu_baseline(wl, line["e2e"]["value"])
        except Exception as e:
            line["torch_gpu_baseline"] = f"failed: {e!r}"
        torch.cuda.empty_cache()
    if world == 1 and not args.no_cpu_baseline:
        try:
            cb = cpu_reference_sample(T, wl.cfg["frame"], unet_iters=3)
            line["cpu_baseline"] = {"value": cb["fps"], "unit": "frames/s", "cores": cb["cores"], "kind": "port",
                                    "sample": cb["sample"]}
        except Exception as e:  # the checker must not take the measurement down
            line["cpu_baseline"] = {"value": None, "unit": "frames/s", "cores": os.cpu_count(), "kind": "port",
                                    "sample": f"failed: {e!r}"}


def torch_gpu_baseline(wl, our_fps):
    """The GPU-LIBRARY line (SURVEY 2.1 / BASELINE.md section 4 "secondary comparison"): the restated reference modules
    (oracle UNet + seg-AE decoder: plain PyTorch, cuDNN convolutions, F.scaled_dot_product_attention) on the SAME B200,
    one batch of 8 frames, 3 DDIM iterations timed after 1 warm-up, frames/s extrapolated to the full schedule + one
    decode. Two settings: the reference's own (fp32, TF32 off: base.yaml:95 allow_tf32 False, weight_dtype float32)
    and the fastest stock option (bf16 autocast). Outside the timed region of the metric; a context number."""
    from oracle import ldmseg_oracle as LO
    from oracle import unet_oracle as UO
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.models import unet_init
    dev, T = wl.env["dev"], wl.T
    B = wl.batch
    unet = UO.build_unet(seed=0, model_kwargs=unet_init.TRAINED_LIKE_MODEL_KWARGS).to(dev)
    vae = LO.build_seg_decoder(seed=1).to(dev)
    UO.USE_SDPA = True
    sched = LO.DDIMOracle()
    sched.set_timesteps_inference(T)
    rgb, lat0 = wl.rgb_dev[:B], wl.noise_dev[:B]
    out = {}
    tf32 = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    try:
        for label, autocast in (("fp32_tf32_off", False), ("bf16_autocast_sdpa", True)):
            torch.backends.cuda.matmul.allow_tf32 = False
            torch.backends.cudnn.allow_tf32 = False
            lat = lat0.clone()
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
                for i in range(4):
                    if i == 1:
                        ev[0].record()
                    t = sched.timesteps[i]
                    eps = unet(torch.cat([lat, rgb], 1), t, encoder_hidden_states=None).float()
                    lat, _ = sched.step(eps, t, lat)
                ev[1].record()
                logits = LO.decode_latents(vae, lat)
                ev[2].record()
            torch.cuda.synchronize()
            ms_iter, ms_dec = ev[0].elapsed_time(ev[1]) / 3, ev[1].elapsed_time(ev[2])
            fps = B / ((T * ms_iter + ms_dec) / 1e3)
            out[label] = {"ms_per_unet_iteration": round(ms_iter, 2), "ms_decode_full_res_logits": round(ms_dec, 2),
                          "frames_per_s": fps, "ours_over_this": our_fps / fps}
            del logits
    finally:
        UO.USE_SDPA = False
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = tf32
    out["note"] = ("oracle modules (restated diffusers UNet + reference seg-AE decoder) in stock PyTorch on this GPU; "
                   "3 DDIM iterations of one 8-frame batch, extrapolated; excludes the ids / merge / PQ tail")
    return out


def run_ours(args):
    import torch.distributed as dist
    from video_latent_diffusion_panoptic_segmentation_b200 import _lib as L
    from video_latent_diffusion_panoptic_segmentation_b200.tools import main_ldm
    world = int(os.environ.get("WORLD_SIZE", 1))
    rank = int(os.environ.get("RANK", 0))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L.lib()  # fails loudly if the CUDA library is missing or the device is not sm_100
    p = copy.deepcopy(main_ldm.BASE)
    env = {"world": world, "rank": rank, "local": local, "dev": dev, "models": main_ldm.build_models(p, dev, seed=0)}
    if args.ln_fold:
        env["models"][1].ln_fold = True   # read when the weights are packed (first forward)
    for name in args.config.split(","):
        run_config(name, args, env)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


_JSON_OUT = None


def emit(line):
    """The JSON line goes to the process's original stdout; everything else that writes to fd 1 (the NCCL version
    banner at N > 1, library prints) has been moved to stderr by main()."""
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="batch8", help="comma-separated subset of " + ", ".join(CONFIGS))
    ap.add_argument("--ddim-steps", type=int, default=50)
    ap.add_argument("--frames-per-gpu", type=int, default=None, help="override (weak-scaling configs)")
    ap.add_argument("--clip-frames", type=int, default=None, help="override the clip length (strong-scaling configs)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-baseline", action="store_true")
    ap.add_argument("--ln-fold", action="store_true", help="A/B: LayerNorm folded into the GEMMs around it instead of its own pass (slower, see DESIGN.md)")
    ap.add_argument("--profile-out", default=None, help="write the per-launch CUDA-event profile of one UNet forward")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write what the last timed step computed (panoptic ids, PQ and DVPQ statistics) to "
                         "DIR/<config>_<array>.npy, at most 64 MB in all; the inputs are seeded, so two builds run with "
                         "the same arguments can be compared array for array")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    for name in args.config.split(","):
        if name not in CONFIGS:
            ap.error(f"unknown config {name!r}")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
