"""B200 mirror of the SAMPLING half of ``TrainerDiffusion`` (ldmseg/trainers/trainers_ldm_cond.py):
``sample`` (:1048-1173), ``decode_latents`` (:398-444), ``crop_padding`` (:1175-1181), ``compute_pq`` (:1184-1375),
``compute_metrics`` (:990-1045). The training half (loss, optimiser, logging, checkpoints) is out of scope.

Data flow of one batch, all on the GPU:
  noise (CPU generator, as the reference) -> H2D
  T x [ UNet CUDA graph (concat+cast fused into conv_in)  ->  fused DDIM (DPM-Solver++, UniPC) update ]    no host sync inside
  seg-AE decoder (NHWC fp32 logits at 4h x 4w)
  fused bilinear x2 + argmax + softmax-max threshold + per-class areas  ->  merge filter  ->  int32 panoptic ids
  PQ / DVPQ statistics from joint id histograms
"""
from typing import Callable, List, Optional

import numpy as np
import torch

from ..evaluations.cityscapes_pap_eval import CityscapesPanopticEvaluator
from ..schedulers import DPMSolverMultistepScheduler, UniPCMultistepScheduler
from ..utils import color_map, get_world_size, is_dist_avail_and_initialized, is_main_process
from ... import _lib as L
from ... import ops

f32, i32 = torch.float32, torch.int32


class TrainerDiffusion:
    def __init__(self, p: dict = None, vae_image=None, vae_semseg=None, unet_model=None, tokenizer=None,
                 text_encoder=None, noise_scheduler=None, image_descriptor_model=None, ema_unet=None, args=None,
                 results_folder=None, save_and_sample_every=1000, cudnn_on=False, fp16=False, ema_on=False,
                 weight_dtype=torch.float32):
        p = p or {}
        self.p = p
        self.args = args or {"gpu": torch.cuda.current_device() if torch.cuda.is_available() else 0}
        self.vae_image, self.vae_semseg, self.unet_model = vae_image, vae_semseg, unet_model
        self.noise_scheduler = noise_scheduler
        # CLIP image / text encoders are third-party models (transformers); when given they are called as the reference
        # calls them (:1102-1122) and only produce the UNet's encoder_hidden_states
        self.image_descriptor_model, self.textencoder, self.tokenizer = image_descriptor_model, text_encoder, tokenizer
        ek = p.get("eval_kwargs", {})
        self.mask_th = ek.get("mask_th", 0.5)
        self.count_th = ek.get("count_th", 512)
        self.overlap_th = ek.get("overlap_th", 0.5)
        tk = p.get("train_kwargs", {})
        self.self_condition = bool(tk.get("self_condition", False))
        self.ignore_label = p.get("ignore_label", 127)
        self.num_classes = p.get("num_classes", 128)
        self.cmap = color_map()   # :173, the palette decode_latents / encode_seg paint label maps with
        self.fp16_scaler = None
        self.weight_dtype = weight_dtype
        self.unet_dtype = torch.float32
        self.latent_size = p.get("latent_size", None)
        self.dl_val = None
        self.best_pq = 0.0
        self.last_results = None
        self.device = torch.device("cuda", self.args["gpu"]) if isinstance(self.args["gpu"], int) else torch.device(
            self.args["gpu"])
        self._loop = {}
        self._stream = {}

    # ------------------------------------------------------------------ encode_inputs (:336-396)
    @torch.no_grad()
    def encode_inputs(self, images, sample_posterior=False, encode_func=None, scaling_factor=None, resize=(192, 640),
                      weight_dtype=None):
        """Images [B,3,H,W] in [0,1] -> (latents, latents_mean), both [B,4,h,w] f32 times the scaling factor:
        optional bilinear resize of the image, ``2 * images - 1`` (fused into the VAE's conv_in), ``encode(...)
        .latent_dist.mode()`` (or ``.sample()``), optional bilinear resize of the latents to ``self.latent_size``
        (an int as in the reference, or an (h, w) pair: SURVEY fact 7)."""
        own = encode_func is None or getattr(encode_func, "__self__", None) is self.vae_image
        if own and self.vae_image is None:
            raise L.LdmError("encode_inputs: no vae_image was given to the trainer")
        if scaling_factor is None:
            scaling_factor = self.vae_image.scaling_factor
        if not images.is_cuda:
            raise L.LdmError("encode_inputs needs CUDA tensors: there is no CPU fallback")
        images = images.contiguous().float()
        if resize is not None and tuple(images.shape[-2:]) != tuple(resize):
            resized = torch.empty(images.shape[:2] + tuple(resize), dtype=f32, device=images.device)
            images = ops.resize_bilinear_planar(images, resized)
        if own:
            from ..models.vae import DiagonalGaussianDistribution
            latent_dist = DiagonalGaussianDistribution(self.vae_image.encode_moments(images, scale=2.0, shift=-1.0))
        else:
            latent_dist = encode_func(2. * images - 1.).latent_dist
        latents_mean = latent_dist.mode()
        latents = latent_dist.sample() if sample_posterior else latents_mean.clone()
        if resize is not None:
            ls = self.latent_size
            if ls is None:
                raise L.LdmError("encode_inputs: resize is set but the trainer has no latent_size (p['latent_size']); "
                                 "pass resize=None to keep the encoder's own latent size")
            size = (int(ls), int(ls)) if isinstance(ls, int) else tuple(int(v) for v in ls)
            if tuple(latents.shape[-2:]) != size:
                def rs(t):
                    out = torch.empty(t.shape[:2] + size, dtype=f32, device=t.device)
                    return ops.resize_bilinear_planar(t.contiguous().float(), out)
                latents, latents_mean = rs(latents), rs(latents_mean)
        return latents * scaling_factor, latents_mean * scaling_factor

    # ------------------------------------------------------------------ sample (:1048-1173)
    def _loop_state(self, B, h, w, multiplier=1, ctx_len=None, dpm=False, unipc_order=0):
        """Static buffers + UNet plan for the DDIM loop at this shape (built once, reused for every batch). With
        classifier-free guidance (multiplier 2) the UNet runs on the doubled batch [uncond | text] (:1129,1126).
        dpm: also the x0_prev buffer of the DPM-Solver++ loop (same plan). unipc_order: also the buffers of the UniPC
        loop at that solver order, the corrected sample `unipc_last` and the x0 history `unipc_hist` (same plan)."""
        key = (B, h, w, self.self_condition, multiplier, ctx_len)
        st = self._loop.get(key)
        if st is None:
            dev, n = self.device, B * multiplier
            st = {"latents": torch.empty((n, 4, h, w), dtype=f32, device=dev),
                  "rgb": torch.empty((n, 4, h, w), dtype=f32, device=dev)}
            parts = [st["latents"], st["rgb"]]
            if self.self_condition:
                st["cond"] = torch.zeros((n, 4, h, w), dtype=f32, device=dev)
                parts.append(st["cond"])
            st["plan"] = self.unet_model._get_plan(n, h, w, 4 * len(parts), parts=parts, ctx_len=ctx_len)
            self._loop[key] = st
        if dpm and "x0_prev" not in st:  # the DPM-Solver++ update's previous x0 prediction
            st["x0_prev"] = torch.empty((B, 4, h, w), dtype=f32, device=self.device)
        if unipc_order:
            if "unipc_last" not in st:
                st["unipc_last"], st["unipc_hist"] = torch.empty((B, 4, h, w), dtype=f32, device=self.device), []
            while len(st["unipc_hist"]) < unipc_order:
                st["unipc_hist"].append(torch.empty((B, 4, h, w), dtype=f32, device=self.device))
        return st

    def norm_resize_images(self, x):
        """:665-677: what the CLIP / DINO descriptor models expect (input of a third-party model: plain torch)."""
        import torch.nn.functional as F
        dev = x.device
        mean_in = torch.tensor([0.485, 0.456, 0.406], device=dev).view(1, 3, 1, 1)
        std_in = torch.tensor([0.229, 0.224, 0.225], device=dev).view(1, 3, 1, 1)
        identifier = self.image_descriptor_model.__class__.__name__.lower()
        if "clip" in identifier:
            x = F.interpolate(x, size=(224, 224), mode="bilinear", align_corners=False)
            mean = torch.tensor([0.48145466, 0.4578275, 0.40821073], device=dev).view(1, 3, 1, 1)
            std = torch.tensor([0.26862954, 0.26130258, 0.27577711], device=dev).view(1, 3, 1, 1)
            return (x - mean) / std
        if "dino" in identifier:
            x = F.interpolate(x, size=(518, 518), mode="bilinear", align_corners=False)
        return (x - mean_in) / std_in

    def _descriptors(self, prompts, rgb_images, batch_size):
        """:1100-1122 -> (encoder_hidden_states of the conditional half, of the unconditional half or None).
        Image descriptors: the reference concatenates the SAME descriptors twice, so both halves of its doubled batch
        are identical and `uncond + g * (text - uncond)` is `uncond` bit for bit: one half is computed here."""
        ctx, uncond = None, None
        if self.image_descriptor_model is not None:
            assert rgb_images is not None
            d = self.image_descriptor_model(self.norm_resize_images(rgb_images).to(self.weight_dtype))["last_feat"]
            ctx = d.view(d.shape[0], d.shape[1], -1).permute(0, 2, 1).to(torch.float)
        if self.textencoder is not None:
            dev = self.device
            ti = self.tokenizer(prompts, padding="max_length", max_length=self.tokenizer.model_max_length,
                                truncation=True, return_tensors="pt")
            ctx = self.textencoder(ti.input_ids.to(device=dev))[0].to(torch.float)
            ui = self.tokenizer([""] * batch_size, padding="max_length", max_length=ti.input_ids.shape[-1],
                                return_tensors="pt")
            uncond = self.textencoder(ui.input_ids.to(device=dev))[0].to(torch.float)
        return ctx, uncond

    @torch.no_grad()
    def sample(self, prompts: List[str], num_inference_steps: int = 50, guidance_scale: float = 7.5,
               seed: Optional[int] = None, rgb_latents: Optional[torch.Tensor] = None,
               return_all_latents: bool = False, disable_progress_bar: bool = False,
               rgb_images: Optional[torch.Tensor] = None, scheduler: Optional[Callable] = None,
               repeat_noise: Optional[bool] = None, noise: Optional[torch.Tensor] = None) -> torch.Tensor:
        if scheduler is None:
            scheduler = self.noise_scheduler
            scheduler.set_timesteps_inference(num_inference_steps)
        dpm = isinstance(scheduler, DPMSolverMultistepScheduler)
        unipc = isinstance(scheduler, UniPCMultistepScheduler)
        if not (dpm or unipc) and not (hasattr(scheduler, "coef_table") and hasattr(scheduler, "clip_range")):
            raise NotImplementedError(f"sample: scheduler {type(scheduler).__name__} is not supported: pass this "
                                      "package's DDIMNoiseScheduler, DPMSolverMultistepScheduler or "
                                      "UniPCMultistepScheduler")
        if dpm and self.self_condition:
            raise NotImplementedError("self_condition with DPMSolverMultistepScheduler: the condition is the step's "
                                      "pred_original_sample (:1152-1153), which the DPM-Solver step output does not carry")
        if unipc and self.self_condition:
            raise NotImplementedError("self_condition with UniPCMultistepScheduler: the condition is the step's "
                                      "pred_original_sample (:1152-1153), which the UniPC step output does not carry")
        if rgb_latents is None:
            raise NotImplementedError("unconditional sampling (rgb_latents=None) is not on the eval path")
        if repeat_noise is None:
            repeat_noise = False
        batch_size = len(prompts) if prompts is not None else rgb_latents.shape[0]
        dev = self.device
        h, w = rgb_latents.shape[-2:]  # SURVEY fact 7: the reference's (latent_size, latent_size) generalised
        if noise is None:
            rng_generator = torch.Generator().manual_seed(seed) if seed is not None else None
            noise = torch.randn((batch_size, 4, h, w), generator=rng_generator)  # CPU generator, as :1091-1094
        if repeat_noise:
            noise = noise[0:1].repeat(batch_size, 1, 1, 1)
        unet = self.unet_model
        ctx, uncond = self._descriptors(prompts, rgb_images, batch_size)
        if ctx is not None and not unet.has_cross_attention():
            ctx = uncond = None  # attn2 is None in every block: the reference's UNet ignores encoder_hidden_states too
        multiplier = 2 if uncond is not None else 1
        if multiplier > 1 and self.self_condition:
            raise NotImplementedError("self_condition with a text encoder: the reference concatenates a doubled batch "
                                      "with an undoubled condition (:1134-1136,1152-1153) and fails")
        B = batch_size
        st = self._loop_state(B, h, w, multiplier, ctx_len=None if ctx is None else ctx.shape[1], dpm=dpm,
                              unipc_order=scheduler.solver_order if unipc else 0)
        lat_all, plan = st["latents"], st["plan"]
        latents = lat_all[:B]
        latents.copy_(noise.to(dev, non_blocking=True))           # H2D (:1095)
        if scheduler.init_noise_sigma != 1.0:
            latents.mul_(scheduler.init_noise_sigma)
        original_noise = latents.clone() if repeat_noise else None
        st["rgb"][:B].copy_(rgb_latents.to(dev, f32))
        if multiplier > 1:
            st["rgb"][B:].copy_(st["rgb"][:B])                    # torch.cat([rgb_latents] * multiplier) (:1126)
        if self.self_condition:
            st["cond"].zero_()
        if ctx is not None:  # k / v of every attn2 layer are projected once here, not once per step
            unet.set_context(plan, ctx if uncond is None else torch.cat([uncond, ctx]))   # (:1120)
        timesteps = scheduler.timesteps.to(dev)
        if dpm:
            return self._dpm_loop(st, latents, B, multiplier, scheduler, timesteps, guidance_scale, return_all_latents,
                                  original_noise)
        if unipc:
            return self._unipc_loop(st, latents, B, multiplier, scheduler, timesteps, guidance_scale,
                                    return_all_latents, original_noise)
        coef = scheduler.coef_table(dev)
        clip = scheduler.clip_range()  # scheduler.step's clip_sample (:1152-1154 calls it with its defaults)
        all_latents = []
        n = timesteps.numel()
        for i in range(n):
            t = timesteps[i:i + 1]
            plan.timestep.copy_(t)                                  # device-side timestep: no host sync in the loop
            if multiplier > 1:
                lat_all[B:].copy_(latents)                          # torch.cat([latents] * multiplier) (:1129)
            if plan.graph is not None:
                plan.graph.replay()                                 # UNet (:1143-1144), concat fused into conv_in
            else:
                unet._run_plan(plan)
            t_index = t.view(torch.int32)[:1]
            last = i == n - 1
            # guidance (:1147-1149) + DDIM update (:1152-1162) in one launch: prev_sample, or pred_original_sample on
            # the last step, written in place
            ops.ddim_step(plan.out[:B], latents, coef, t_index,
                          prev_sample=None if last else latents,
                          pred_x0=latents if last else (st["cond"] if self.self_condition else None),
                          eps_text=plan.out[B:] if multiplier > 1 else None, guidance_scale=guidance_scale,
                          clip_sample_range=clip)
            if return_all_latents:
                all_latents.append(latents.clone())
        if return_all_latents:
            return torch.cat(all_latents, dim=0)
        out = latents.clone()
        if repeat_noise:
            return out, original_noise
        return out

    def _dpm_loop(self, st, latents, B, multiplier, scheduler, timesteps, guidance_scale, return_all_latents,
                  original_noise):
        """The sampler loop of sample() with a DPMSolverMultistepScheduler: the same UNet graph, then one fused
        DPM-Solver++ update (guidance included) per step. Its last step goes to sigma = 0, where prev equals x0: the
        latents end as the final x0 prediction, as DDIM's last step leaves them."""
        dev, lat_all, plan = self.device, st["latents"], st["plan"]
        coef, steps = scheduler.coef_table(dev), scheduler.step_index_table(dev)
        x0_prev = st["x0_prev"]
        all_latents = []
        for i in range(timesteps.numel()):
            plan.timestep.copy_(timesteps[i:i + 1])
            if multiplier > 1:
                lat_all[B:].copy_(latents)
            if plan.graph is not None:
                plan.graph.replay()
            else:
                self.unet_model._run_plan(plan)
            ops.dpmpp_step(plan.out[:B], latents, coef, steps[i:i + 1], prev_sample=latents, x0_prev=x0_prev,
                           eps_text=plan.out[B:] if multiplier > 1 else None, guidance_scale=guidance_scale)
            if return_all_latents:
                all_latents.append(latents.clone())
        if return_all_latents:
            return torch.cat(all_latents, dim=0)
        out = latents.clone()
        if original_noise is not None:
            return out, original_noise
        return out

    def _unipc_loop(self, st, latents, B, multiplier, scheduler, timesteps, guidance_scale, return_all_latents,
                    original_noise):
        """The sampler loop of sample() with a UniPCMultistepScheduler: the same UNet graph, then one fused UniPC
        update (guidance, corrector of the previous step, predictor, history shift) per step. Its last step goes to
        sigma = 0, where prev equals the final x0 prediction, as DDIM's last step leaves the latents."""
        dev, lat_all, plan = self.device, st["latents"], st["plan"]
        coef, steps = scheduler.coef_table(dev), scheduler.step_index_table(dev)
        last, hist = st["unipc_last"], st["unipc_hist"][:scheduler.solver_order]
        all_latents = []
        for i in range(timesteps.numel()):
            plan.timestep.copy_(timesteps[i:i + 1])
            if multiplier > 1:
                lat_all[B:].copy_(latents)
            if plan.graph is not None:
                plan.graph.replay()
            else:
                self.unet_model._run_plan(plan)
            ops.unipc_step(plan.out[:B], latents, coef, steps[i:i + 1], prev_sample=latents, last=last, history=hist,
                           eps_text=plan.out[B:] if multiplier > 1 else None, guidance_scale=guidance_scale)
            if return_all_latents:
                all_latents.append(latents.clone())
        if return_all_latents:
            return torch.cat(all_latents, dim=0)
        out = latents.clone()
        if original_noise is not None:
            return out, original_noise
        return out

    # ------------------------------------------------------------------ streaming sampler
    def sample_stream(self, frames, num_inference_steps, scheduler=None, batch_size=8, seed=None):
        """Sample a stream of frames through `batch_size` slots: every UNet forward advances each occupied slot by one
        step of its own trajectory, a finished frame leaves its slot and the next frame takes it in the same forward.
        That is the throughput of batch `batch_size` at a latency of N forwards per frame.

        frames: iterable of (frame_id, rgb_latents [1,4,h,w], noise [1,4,h,w] or None); noise None is drawn from a CPU
        generator seeded seed + frame_id (stream_noise). An item None means that no frame has arrived yet: the free
        slots stay empty for that forward. Returns a generator of (frame_id, final latents [1,4,h,w]) in finishing
        order. A frame's latents equal, bit for bit, those sample() gives it in a batch of `batch_size` at the same
        position with the same noise. All frames take the same N; classifier-free guidance, self_condition, a
        per-frame cross-attention context and DDIM's clip_sample are not built (learnable object queries are: their
        context is the same for every frame)."""
        if self.self_condition:
            raise NotImplementedError("sample_stream: self_condition (the condition is each step's x0 prediction, "
                                      "which the streaming updates do not carry)")
        if self.textencoder is not None:
            raise NotImplementedError("sample_stream: classifier-free guidance (a text encoder doubles the batch into "
                                      "unconditional and conditional halves)")
        if self.image_descriptor_model is not None and self.unet_model.has_cross_attention():
            raise NotImplementedError("sample_stream: a cross-attention context that differs per frame (image "
                                      "descriptors); learnable object queries are supported")
        if scheduler is None:
            scheduler = self.noise_scheduler
            scheduler.set_timesteps_inference(num_inference_steps)
        dpm = isinstance(scheduler, DPMSolverMultistepScheduler)
        unipc = isinstance(scheduler, UniPCMultistepScheduler)
        if not (dpm or unipc) and not (hasattr(scheduler, "coef_table") and hasattr(scheduler, "clip_range")):
            raise NotImplementedError(f"sample_stream: scheduler {type(scheduler).__name__} is not supported: pass this "
                                      "package's DDIMNoiseScheduler, DPMSolverMultistepScheduler or "
                                      "UniPCMultistepScheduler")
        if not (dpm or unipc) and scheduler.clip_range() != 0.0:
            raise NotImplementedError("sample_stream: DDIM with clip_sample")
        if batch_size < 1:
            raise ValueError(f"sample_stream: batch_size={batch_size}")
        return self._stream_loop(frames, scheduler, "dpm" if dpm else "unipc" if unipc else "ddim", batch_size, seed)

    def _stream_state(self, B, h, w, kind, order):
        """Static buffers of the streaming loop at this shape, and the UNet's per-image-timestep plan reading them."""
        key = (B, h, w, kind, order)
        st = self._stream.get(key)
        if st is None:
            dev = self.device
            z = lambda: torch.zeros((B, 4, h, w), dtype=f32, device=dev)  # noqa: E731
            st = {"latents": z(), "rgb": z(), "rows": torch.zeros((B,), dtype=i32, device=dev)}
            st["plan"] = self.unet_model._get_plan(B, h, w, 8, parts=[st["latents"], st["rgb"]], per_image_t=True)
            # host side of the per-forward copies, one set per forward in flight (see _stream_loop)
            st["ts_host"] = torch.zeros((2, B), dtype=torch.int64).pin_memory()
            st["rows_host"] = torch.zeros((2, B), dtype=i32).pin_memory()
            st["noise_host"] = torch.zeros((2, B, 4, h, w), dtype=f32).pin_memory()
            st["done"] = [torch.cuda.Event(), torch.cuda.Event()]
            if kind == "ddim":
                st["x0"] = z()             # the last step's result is its x0 prediction, as in sample()
            elif kind == "dpm":
                st["x0_prev"] = z()
            else:
                st["last"], st["hist"] = z(), [z() for _ in range(order)]
            self._stream[key] = st
        return st

    @torch.no_grad()
    def _stream_loop(self, frames, scheduler, kind, B, seed):
        dev = self.device
        timesteps = scheduler.timesteps.cpu().tolist()
        N = len(timesteps)
        coef = scheduler.coef_table(dev)
        st, plan = None, None
        for admitted, steps, finished in stream_schedule(frames, N, B):
            if st is None:
                h, w = admitted[0][1][1].shape[-2:]
                st = self._stream_state(B, h, w, kind, scheduler.solver_order if kind == "unipc" else 0)
                plan, lat, rgb, rows = st["plan"], st["latents"], st["rgb"], st["rows"]
                fwd = 0
            # The loop reads nothing back from the device: rows and timesteps go host -> device, a finished frame's
            # latents are cloned on the device. Its one wait is on the forward before the previous one, which keeps the
            # GPU one forward ahead of admission (a frame that arrives while a forward runs joins the next one) and
            # frees that forward's set of pinned host buffers for reuse.
            ring = fwd % 2
            fwd += 1
            st["done"][ring].synchronize()
            ts_h, rows_h, noise_h = st["ts_host"][ring], st["rows_host"][ring], st["noise_host"][ring]
            for s, (fid, rgb_f, noise) in admitted:
                noise_h[s].copy_((noise if noise is not None else stream_noise(fid, seed, lat.shape[1:])).reshape(
                    lat.shape[1:]))
                lat[s].copy_(noise_h[s], non_blocking=True)
                if scheduler.init_noise_sigma != 1.0:
                    lat[s].mul_(scheduler.init_noise_sigma)
                rgb[s].copy_(rgb_f.reshape(rgb.shape[1:]).to(dev, f32), non_blocking=True)
            for s, i in enumerate(steps):
                if i is None:               # an empty slot runs step 0 on zeros; its result is never read
                    lat[s].zero_()
                    rgb[s].zero_()
                i = 0 if i is None else i
                ts_h[s] = timesteps[i]
                rows_h[s] = timesteps[i] if kind == "ddim" else i
            plan.timesteps.copy_(ts_h, non_blocking=True)
            rows.copy_(rows_h, non_blocking=True)
            if plan.graph is not None:
                plan.graph.replay()
            else:
                self.unet_model._run_plan(plan)
            epi = lat[0].numel()
            if kind == "ddim":
                ops.ddim_step_rows(plan.out, lat, coef, rows, epi, prev_sample=lat, pred_x0=st["x0"])
            elif kind == "dpm":
                ops.dpmpp_step_rows(plan.out, lat, coef, rows, epi, prev_sample=lat, x0_prev=st["x0_prev"])
            else:
                ops.unipc_step_rows(plan.out, lat, coef, rows, epi, prev_sample=lat, last=st["last"],
                                    history=st["hist"])
            st["done"][ring].record()
            final = st["x0"] if kind == "ddim" else lat   # DPM-Solver++ / UniPC end at sigma = 0, where prev is x0
            for s, (fid, _, _) in finished:
                yield fid, final[s:s + 1].clone()

    # ------------------------------------------------------------------ decode_latents (:398-444)
    @torch.no_grad()
    def decode_latents(self, latents, return_logits=False, threshold_output=False, rgb_latents=None,
                       weight_dtype=torch.float32):
        logits = self.vae_semseg.decode_nhwc(latents, scale=1.0 / self.vae_semseg.scaling_factor)
        up = self.vae_semseg.interpolation_factor
        B, H, W, C = logits.shape
        if return_logits:
            images = torch.empty((B, C, H * up, W * up), dtype=f32, device=logits.device)
            ops.bilinear_up_nchw(logits, images, up)
            return images
        ids = torch.empty((B, H * up, W * up), dtype=i32, device=logits.device)
        counts = torch.empty((B, 2, C), dtype=i32, device=logits.device)
        ops.logits_to_ids(logits, ids, counts, up=up, mask_th=self.mask_th if threshold_output else -1.0,
                          ignore_label=self.ignore_label)
        # :435-436: the label map leaves as a colour image, uint8 [B, H, W, 3]
        return self.encode_seg(ids.cpu().numpy()).astype(np.uint8)

    def encode_seg(self, semseg, cmap=None):
        """trainers_ldm_cond.py:326-334: labels [B, H, W] (taken modulo 256, as the reference's astype(uint8) does) ->
        the palette colour of every pixel, [B, H, W, cmap.shape[1]] in the palette's dtype. One gather instead of the
        reference's loop over the labels present."""
        if cmap is None:
            if getattr(self, "cmap", None) is None:
                self.cmap = color_map()
            cmap = self.cmap
        return cmap[np.asarray(semseg).astype(np.uint8)]

    @torch.no_grad()
    def panoptic_ids(self, latents):
        """Fused tail (:1255-1325 with identity resizes): latents -> (ids before the merge, cleaned ids with -1 = void,
        per-class [argmax area, sigmoid area]) as int32 device tensors."""
        logits = self.vae_semseg.decode_nhwc(latents, scale=1.0 / self.vae_semseg.scaling_factor)
        up = self.vae_semseg.interpolation_factor
        B, H, W, C = logits.shape
        ids = torch.empty((B, H * up, W * up), dtype=i32, device=logits.device)
        counts = torch.empty((B, 2, C), dtype=i32, device=logits.device)
        ops.logits_to_ids(logits, ids, counts, up=up, mask_th=self.mask_th, ignore_label=self.ignore_label)
        cleaned = torch.empty_like(ids)
        ops.segment_filter(ids, counts, cleaned, count_th=self.count_th, overlap_th=self.overlap_th,
                           ignore_label=self.ignore_label)
        return ids, cleaned, counts

    @torch.no_grad()
    def panoptic_ids_resized(self, latents, rgb_size, padding_masks=None, im_sizes=None):
        """General tail (:1255-1325) for the cases where the resizes are not the identity: decoder logits ->
        bilinear x interpolation_factor (vae.py:271) -> bilinear to the RGB size (:1264-1269) -> per image
        crop_padding (:1175-1181) -> bilinear to meta.im_size (:1279-1284) -> argmax / threshold / merge.
        Returns a list of (ids, cleaned, counts) int32 device tensors, one entry per image ([1, h_i, w_i])."""
        logits = self.vae_semseg.decode_nhwc(latents, scale=1.0 / self.vae_semseg.scaling_factor)
        up = self.vae_semseg.interpolation_factor
        B, H, W, C = logits.shape
        dev = logits.device
        full = torch.empty((B, H * up, W * up, C), dtype=f32, device=dev)
        ops.resize_bilinear_nhwc(logits, full)
        rh, rw = int(rgb_size[0]), int(rgb_size[1])
        if (rh, rw) != (H * up, W * up):
            full2 = torch.empty((B, rh, rw, C), dtype=f32, device=dev)
            ops.resize_bilinear_nhwc(full, full2)
            full = full2
        out = []
        for b in range(B):
            if padding_masks is not None:
                y0, y1, x0, x1 = self.crop_padding_box(padding_masks[b])
            else:
                y0, y1, x0, x1 = 0, rh - 1, 0, rw - 1
            oh, ow = (int(im_sizes[b][0]), int(im_sizes[b][1])) if im_sizes is not None else (y1 - y0 + 1, x1 - x0 + 1)
            img = torch.empty((1, oh, ow, C), dtype=f32, device=dev)
            ops.resize_bilinear_nhwc(full[b:b + 1], img, crop=(y0, x0, y1 - y0 + 1, x1 - x0 + 1))
            ids = torch.empty((1, oh, ow), dtype=i32, device=dev)
            counts = torch.empty((1, 2, C), dtype=i32, device=dev)
            ops.logits_to_ids(img, ids, counts, up=1, mask_th=self.mask_th, ignore_label=self.ignore_label)
            cleaned = torch.empty_like(ids)
            ops.segment_filter(ids, counts, cleaned, count_th=self.count_th, overlap_th=self.overlap_th,
                               ignore_label=self.ignore_label)
            out.append((ids, cleaned, counts))
        return out

    @staticmethod
    def crop_padding_box(padding_mask):
        """Bounding box (y0, y1, x0, x1, inclusive) of the non-zero padding mask, as crop_padding (:1175-1181)."""
        rows = padding_mask.to(torch.bool).any(dim=1).nonzero()
        cols = padding_mask.to(torch.bool).any(dim=0).nonzero()
        box = torch.stack([rows.min(), rows.max(), cols.min(), cols.max()]).cpu().tolist()
        return int(box[0]), int(box[1]), int(box[2]), int(box[3])

    def crop_padding(self, prediction, padding_mask):
        co = padding_mask.nonzero()
        y0, y1 = co[:, 0].min(), co[:, 0].max()
        x0, x1 = co[:, 1].min(), co[:, 1].max()
        return prediction[:, y0:y1 + 1, x0:x1 + 1]

    # ------------------------------------------------------------------ compute_pq (:1184-1375)
    @torch.no_grad()
    def compute_pq(self, num_inference_steps=50, guidance_scale=7.5, seed=None, threshold_output=True,
                   save_images=False, max_iter=None, dataloader=None, threshold_mode="max", save_model=False):
        """`dataloader` yields dicts with 'rgb_latents' [B,4,h,w], or 'image' [B,3,H,W] in [0,1] that goes through the
        RGB VAE encoder first (:1234-1239, SURVEY section 8(f) rank 1), 'semseg' ground-truth labels ([B,H,W], or a list of per-image [h_i,w_i] maps at
        meta.im_size), optional 'mask' [B,Hrgb,Wrgb] padding masks (their size is the RGB input size) and 'meta'
        (per image {'im_size': (h_i, w_i)}). When every resize / crop of :1264-1284 is the identity the fused tail runs;
        otherwise the logits are resized, cropped and resized again as the reference does."""
        if threshold_mode != "max" or not threshold_output:
            raise NotImplementedError("only threshold_mode='max' with threshold_output=True is built")
        if is_main_process():
            print("Computing PQ metric for Cityscapes ...")
        dataloader = dataloader if dataloader is not None else self.dl_val
        thing_ids = {11, 12, 13, 14, 15, 16, 17, 18}
        evaluator = CityscapesPanopticEvaluator(thing_ids=thing_ids, device=self.device)
        evaluator.reset()
        scheduler = self.noise_scheduler
        scheduler.set_timesteps_inference(num_inference_steps=num_inference_steps)
        scheduler.move_timesteps_to(self.device)
        all_cleaned = []
        for batch_idx, data in enumerate(dataloader):
            if "rgb_latents" in data:
                rgb_latents = data["rgb_latents"].to(self.device)
            else:  # :1234-1239: frames go through the RGB VAE encoder first
                if self.vae_image is None or "image" not in data:
                    raise L.LdmError("compute_pq: the batch has no 'rgb_latents'; pass 'image' batches and a vae_image "
                                     "(GeneralVAEImage) to the trainer")
                rgb_latents, _ = self.encode_inputs(data["image"].to(self.device), encode_func=self.vae_image.encode,
                                                    scaling_factor=self.vae_image.scaling_factor,
                                                    resize=p_get(self.p, "rgb_size"))
            gt_semseg = data["semseg"]  # [B,H,W] tensor, or a list of [h_i,w_i] tensors (original image sizes)
            gt_semseg = ([g.to(self.device) for g in gt_semseg] if isinstance(gt_semseg, (list, tuple))
                         else gt_semseg.to(self.device))
            B = rgb_latents.shape[0]
            rgb_images = data["image"].to(self.device) if "image" in data else None
            prompts = list(data["text"]) if "text" in data else [""] * B     # :1241-1252: text= and rgb_images=
            latents = self.sample(prompts, num_inference_steps, guidance_scale, seed, rgb_latents=rgb_latents,
                                  scheduler=scheduler, disable_progress_bar=True, rgb_images=rgb_images)
            f = self.vae_semseg.downsample_factor
            dec_size = (rgb_latents.shape[-2] * f, rgb_latents.shape[-1] * f)
            masks = data["mask"].to(self.device) if "mask" in data else None
            # :1264-1269: the logits are resized to the size of the RGB input
            rgb_size = (tuple(rgb_images.shape[-2:]) if rgb_images is not None
                        else tuple(masks.shape[-2:]) if masks is not None else dec_size)
            im_sizes = [tuple(m["im_size"]) for m in data["meta"]] if "meta" in data else [rgb_size] * B
            identity = (rgb_size == dec_size and all(tuple(sz) == rgb_size for sz in im_sizes)
                        and (masks is None or bool(masks.to(torch.bool).all())))
            if identity:  # every resize / crop of :1264-1284 is the identity: fused tail
                ids, cleaned, _ = self.panoptic_ids(latents)
                evaluator.add_images(cleaned, gt_semseg if torch.is_tensor(gt_semseg) else torch.stack(list(gt_semseg)))
                all_cleaned.append(cleaned)
            else:
                per_image = self.panoptic_ids_resized(latents, rgb_size, masks, im_sizes)
                for b, (_, cleaned, _) in enumerate(per_image):
                    gt_b = gt_semseg[b]
                    if tuple(gt_b.shape[-2:]) != tuple(cleaned.shape[-2:]):
                        raise ValueError(f"ground truth {tuple(gt_b.shape[-2:])} does not match meta.im_size "
                                         f"{tuple(cleaned.shape[-2:])} of image {b}")
                    evaluator.add_image(cleaned[0], gt_b.contiguous())
                    all_cleaned.append(cleaned)
            if max_iter is not None and batch_idx > max_iter:
                break
        self.last_cleaned = all_cleaned
        # the reference never reduces PQ across ranks (SURVEY fact 9); with a process group we all-reduce the
        # integer statistics exactly and gather the float64 IoU sums in rank order
        if is_dist_avail_and_initialized() and get_world_size() > 1:
            reduce_evaluator_(evaluator, self.device)
        results = evaluator.evaluate()
        self.last_results = results
        if is_main_process():
            print(f"Panoptic Quality (PQ): {results['pq']:.2f}")
            print(f"Segmentation Quality (SQ): {results['sq']:.2f}")
            print(f"Recognition Quality (RQ): {results['rq']:.2f}")
            if "thing_pq" in results:
                print(f"Things PQ: {results['thing_pq']:.2f}")
                print(f"Stuff PQ: {results['stuff_pq']:.2f}")
        return

    @torch.no_grad()
    def compute_metrics(self, metrics=("pq",), threshold_output=True, save_images=False, seed=None, max_iter=None,
                        dataloader=None, models_to_eval=None, num_inference_steps=50, **kwargs):
        for m in metrics:
            if m != "pq":
                raise NotImplementedError(f"metric {m} is not on the sampling path")
            self.compute_pq(num_inference_steps=num_inference_steps, seed=seed, threshold_output=threshold_output,
                            save_images=save_images, max_iter=max_iter, dataloader=dataloader)
        if is_dist_avail_and_initialized():
            torch.distributed.barrier()
        return self.last_results


def stream_noise(frame_id, seed, shape):
    """The initial noise of stream frame `frame_id` when it brings none: a CPU generator seeded seed + frame_id (the
    default generator without a seed), shape [4, h, w]."""
    gen = torch.Generator().manual_seed(seed + frame_id) if seed is not None else None
    return torch.randn((1,) + tuple(shape), generator=gen)


def stream_schedule(frames, num_steps, num_slots):
    """Slot bookkeeping of TrainerDiffusion.sample_stream. Yields once per UNet forward (admitted, steps, finished):
      admitted: [(slot, item)], the frames that enter a free slot at this forward, in arrival order (lowest free slot
                first); a frame runs step 0 in the forward it enters;
      steps:    per slot, the step it runs at this forward, or None for an empty slot;
      finished: [(slot, item)], the frames whose last step this forward runs, in arrival order.
    `frames` is pulled only while a slot is free. An item None means nothing has arrived yet: the remaining free slots
    stay empty for this forward, and no forward is yielded while every slot is empty."""
    it = iter(frames)
    item, step = [None] * num_slots, [0] * num_slots
    exhausted = False
    while True:
        admitted = []
        for s in range(num_slots):
            if exhausted or item[s] is not None:
                continue
            try:
                nxt = next(it)
            except StopIteration:
                exhausted = True
                continue
            if nxt is None:
                break
            item[s], step[s] = nxt, 0
            admitted.append((s, nxt))
        if all(x is None for x in item):
            if exhausted:
                return
            continue
        # slots are filled lowest first, so within one forward slot order is arrival order
        finished = [(s, item[s]) for s in range(num_slots) if item[s] is not None and step[s] == num_steps - 1]
        yield admitted, [step[s] if item[s] is not None else None for s in range(num_slots)], finished
        for s in range(num_slots):
            if item[s] is not None:
                step[s] += 1
                if step[s] == num_steps:
                    item[s] = None


def p_get(p, key):
    """`self.rgb_size` of the reference trainer (:159): p['transformation_kwargs']['size_rgb'], an int that
    F.interpolate takes for both dims (:369), or an (h, w) pair here; None = no resize. p['rgb_size'] overrides."""
    if key in p:
        size = p[key]
    else:
        size = p.get("transformation_kwargs", {}).get("size_rgb") if key == "rgb_size" else None
    return (size, size) if isinstance(size, int) else size


def reduce_evaluator_(evaluator, device):
    """Cross-rank reduction of a CityscapesPanopticEvaluator (pattern: SemsegMeter.synchronize_between_processes,
    ldmseg/evaluations/semseg_evaluation.py:59-70). Integers (TP/FP/FN, per class) are all-reduced exactly; the
    float64 IoU sums are all-gathered and added in rank order so the result does not depend on reduction order."""
    import torch.distributed as dist
    backend_dev = device if dist.get_backend() == "nccl" else torch.device("cpu")
    ncls = 256
    ints = torch.zeros((3, ncls + 1), dtype=torch.int64, device=backend_dev)
    ious = torch.zeros((ncls + 1,), dtype=torch.float64, device=backend_dev)
    seen = torch.zeros((ncls,), dtype=torch.int64, device=backend_dev)
    ints[0, ncls], ints[1, ncls], ints[2, ncls] = evaluator.TP, evaluator.FP, evaluator.FN
    ious[ncls] = evaluator.iou_sum
    for c, v in evaluator.TP_per_class.items():
        ints[0, c] = v
        seen[c] = 1
    for c, v in evaluator.FP_per_class.items():
        ints[1, c] = v
    for c, v in evaluator.FN_per_class.items():
        ints[2, c] = v
    for c, v in evaluator.iou_sum_per_class.items():
        ious[c] = v
    dist.all_reduce(ints, op=dist.ReduceOp.SUM)
    dist.all_reduce(seen, op=dist.ReduceOp.SUM)
    gathered = [torch.zeros_like(ious) for _ in range(dist.get_world_size())]
    dist.all_gather(gathered, ious)
    tot = torch.zeros_like(ious)
    for g in gathered:  # rank order
        tot = tot + g
    ints, tot, seen = ints.cpu(), tot.cpu(), seen.cpu()
    evaluator.TP, evaluator.FP, evaluator.FN = int(ints[0, ncls]), int(ints[1, ncls]), int(ints[2, ncls])
    evaluator.iou_sum = float(tot[ncls])
    evaluator.TP_per_class = {c: int(ints[0, c]) for c in range(ncls) if seen[c] > 0}
    evaluator.FP_per_class = {c: int(ints[1, c]) for c in range(ncls) if seen[c] > 0 or ints[1, c] > 0}
    evaluator.FN_per_class = {c: int(ints[2, c]) for c in range(ncls) if seen[c] > 0}
    evaluator.iou_sum_per_class = {c: float(tot[c]) for c in range(ncls) if seen[c] > 0}
    return evaluator
