"""B200 host mirror of ``DDIMNoiseScheduler`` (ldmseg/schedulers/ddim_scheduler.py:26-291).

The schedule (betas, alphas_cumprod, timesteps, loss weights) is built on the host in fp32 exactly like the
reference (:51-95,119-131). ``step`` (:218-269) runs as ONE fused kernel (ldm_ddim_step) that reads the four
per-timestep coefficients from a device table indexed by the timestep value itself, so a CUDA-tensor timestep never
has to be synchronised back to the host (the reference indexes a CPU tensor with it, SURVEY fact 8). The kernel
keeps the reference's op order with round-to-nearest intrinsics: fp32 results are bit-identical to the reference
scheduler running on the CPU.
"""
import math
from typing import Optional, Union

import numpy as np
import torch

from ..utils import OutputDict
from ... import _lib as L
from ... import ops


class DDIMNoiseSchedulerOutput(OutputDict):
    prev_sample: torch.Tensor
    pred_original_sample: Optional[torch.Tensor] = None


def betas_for_alpha_bar(num_diffusion_timesteps, max_beta=0.999) -> torch.Tensor:
    def alpha_bar(t):
        return math.cos((t + 0.008) / 1.008 * math.pi / 2) ** 2
    n = num_diffusion_timesteps
    return torch.tensor([min(1 - alpha_bar((i + 1) / n) / alpha_bar(i / n), max_beta) for i in range(n)],
                        dtype=torch.float32)


def make_betas(beta_schedule: str, beta_start: float, beta_end: float, num_train_timesteps: int,
               owner=None) -> torch.Tensor:
    """The beta schedule (:51-61) in fp32, shared by every scheduler of the package."""
    if beta_schedule == "linear":
        return torch.linspace(beta_start, beta_end, num_train_timesteps, dtype=torch.float32)
    if beta_schedule == "scaled_linear":
        return torch.linspace(beta_start ** 0.5, beta_end ** 0.5, num_train_timesteps, dtype=torch.float32) ** 2
    if beta_schedule == "squaredcos_cap_v2":
        return betas_for_alpha_bar(num_train_timesteps)
    if beta_schedule == "sigmoid":
        return torch.sigmoid(torch.linspace(-6, 6, num_train_timesteps)) * (beta_end - beta_start) + beta_start
    raise NotImplementedError(f"{beta_schedule} does is not implemented for {owner}")


class DDIMNoiseScheduler(object):
    def __init__(self, num_train_timesteps: int = 1000, beta_start: float = 0.0001, beta_end: float = 0.02,
                 beta_schedule: str = "linear", clip_sample: bool = True, set_alpha_to_one: bool = True,
                 steps_offset: int = 0, prediction_type: str = "epsilon", thresholding: bool = False,
                 dynamic_thresholding_ratio: float = 0.995, clip_sample_range: float = 1.0,
                 sample_max_value: float = 1.0, weight: str = "none", max_snr: float = 5.0,
                 device: Union[str, torch.device] = None, verbose: bool = True):
        self.betas = make_betas(beta_schedule, beta_start, beta_end, num_train_timesteps, owner=self.__class__)
        self.alphas = 1.0 - self.betas
        self.alphas_cumprod = torch.cumprod(self.alphas, dim=0)
        self.final_alpha_cumprod = torch.tensor(1.0) if set_alpha_to_one else self.alphas_cumprod[0]
        self.compute_loss_weights(mode=weight, max_snr=max_snr)
        self.weights = self.weights.to(device)
        self.num_train_timesteps = num_train_timesteps
        self.num_inference_steps = None
        self.timesteps = torch.from_numpy(np.arange(0, num_train_timesteps)[::-1].copy().astype(np.int64))
        self.clip_sample, self.clip_sample_range = clip_sample, clip_sample_range
        self.prediction_type = prediction_type
        self.thresholding, self.dynamic_thresholding_ratio = thresholding, dynamic_thresholding_ratio
        self.steps_offset = steps_offset
        self.beta_schedule, self.beta_start, self.beta_end = beta_schedule, beta_start, beta_end
        self.init_noise_sigma = 1.0
        self.verbose = verbose
        self._coef_dev = {}  # device -> f32 [num_train_timesteps, 4]

    def compute_loss_weights(self, mode="max_clamp_snr", max_snr=5.0):
        assert mode in ["inverse_log_snr", "max_clamp_snr", "linear", "fixed", "none"]
        self.weight_mode = mode
        snr = self.alphas_cumprod / (1 - self.alphas_cumprod)
        if mode == "inverse_log_snr":
            self.weights = torch.log(1. / snr).clamp(min=1)
            self.weights /= self.weights[-1]
        elif mode == "max_clamp_snr":
            self.weights = snr.clamp(max=max_snr) / snr
        elif mode == "fixed":
            self.weights = snr
            self.weights[:len(self.weights) // 4] = 0.1
        elif mode == "linear":
            self.weights = torch.arange(1, len(snr) + 1) / len(snr)
        else:
            self.weights = torch.ones_like(snr)

    def get_betas_for_alpha_bar(self, num_diffusion_timesteps, max_beta=0.999) -> torch.Tensor:
        return betas_for_alpha_bar(num_diffusion_timesteps, max_beta)

    # ------------------------------------------------------------------ inference timesteps (:119-136)
    def set_timesteps_inference(self, num_inference_steps: int, device: Union[str, torch.device] = None, tmin: int = 0):
        self.num_inference_steps = num_inference_steps
        step_ratio = self.num_train_timesteps // self.num_inference_steps
        self.steps_offset = step_ratio - 1
        timesteps = (np.arange(0, num_inference_steps) * step_ratio).round()[::-1].copy().astype(np.int64)
        self.timesteps = torch.from_numpy(timesteps).to(device)
        self.timesteps += self.steps_offset
        self.timesteps = self.timesteps[self.timesteps >= tmin]
        self._coef_dev = {}

    def move_timesteps_to(self, device: Union[str, torch.device]):
        self.timesteps = self.timesteps.to(device)

    def step_coefficients(self) -> torch.Tensor:
        """f32 [num_train_timesteps, 4] rows {sqrt(1-a_t), sqrt(a_t), sqrt(a_prev), sqrt(1-a_prev)} with
        prev_t = t - num_train_timesteps // num_inference_steps, built with the reference's own fp32 tensor ops
        (:231-236,240,264,267)."""
        ratio = self.num_train_timesteps // self.num_inference_steps
        a_t = self.alphas_cumprod.to(torch.float32)
        # alphas_cumprod[t - ratio], final_alpha_cumprod where t - ratio < 0: one vectorised pass (the element-wise fp32
        # ops are the ones the reference applies to 0-dim tensors: same bits, checked in tests/test_host_cpu.py)
        a_prev = torch.cat([self.final_alpha_cumprod.to(torch.float32).reshape(1).expand(min(ratio, a_t.numel())),
                            a_t[:max(a_t.numel() - ratio, 0)]])
        return torch.stack([(1 - a_t) ** 0.5, a_t ** 0.5, a_prev ** 0.5, (1 - a_prev) ** 0.5], dim=1).contiguous()

    def coef_table(self, device) -> torch.Tensor:
        device = torch.device(device)
        if device not in self._coef_dev:
            self._coef_dev[device] = self.step_coefficients().to(device)
        return self._coef_dev[device]

    def clip_range(self) -> float:
        """clip_sample_range when clip_sample is on (:253-257), else 0 (= no clipping for ldm_ddim_step_clip)."""
        if not self.clip_sample:
            return 0.0
        if not self.clip_sample_range > 0:
            raise L.LdmError(f"clip_sample needs clip_sample_range > 0, got {self.clip_sample_range}")
        return float(self.clip_sample_range)

    # ------------------------------------------------------------------ step (:218-269)
    def step(self, model_output: torch.Tensor, timestep, sample: torch.Tensor,
             use_clipped_model_output: bool = False) -> DDIMNoiseSchedulerOutput:
        if self.prediction_type != "epsilon":
            raise NotImplementedError("only prediction_type='epsilon' is built (base.yaml:49)")
        if self.thresholding:
            raise NotImplementedError
        if not (model_output.is_cuda and sample.is_cuda):
            raise L.LdmError("DDIMNoiseScheduler.step needs CUDA tensors: there is no CPU fallback")
        dev = sample.device
        coef = self.coef_table(dev)
        if torch.is_tensor(timestep) and timestep.is_cuda:
            # low 32 bits of the int64 timestep (little endian) are the row index: no device->host sync
            t_index = timestep.reshape(-1)[:1].to(torch.int64).contiguous().view(torch.int32)[:1]
        else:
            t_index = torch.tensor([int(timestep)], dtype=torch.int32, device=dev)
        eps = model_output.contiguous().float()
        x = sample.contiguous().float()
        prev, x0 = torch.empty_like(x), torch.empty_like(x)
        ops.ddim_step(eps, x, coef, t_index, prev, x0, clip_sample_range=self.clip_range(),
                      use_clipped_model_output=use_clipped_model_output)
        return DDIMNoiseSchedulerOutput(prev_sample=prev, pred_original_sample=x0)

    # ------------------------------------------------------------------ training-side helpers (:155-216), plain tensor math
    def add_noise(self, original_samples, noise, timesteps, scale: float = 1.0, mask_noise_perc=None):
        ac = self.alphas_cumprod.to(device=original_samples.device, dtype=original_samples.dtype)
        timesteps = timesteps.to(original_samples.device)
        shape = (-1,) + (1,) * (original_samples.dim() - 1)
        sa = (ac[timesteps] ** 0.5).flatten().view(shape)
        sb = ((1 - ac[timesteps]) ** 0.5).flatten().view(shape)
        if mask_noise_perc is not None:
            noise *= torch.rand_like(original_samples) < mask_noise_perc
        return sa * scale * original_samples + sb * noise

    @torch.no_grad()
    def remove_noise(self, noisy_samples, noise, timesteps, scale: float = 1.0):
        ac = self.alphas_cumprod.to(device=noisy_samples.device, dtype=noisy_samples.dtype)
        timesteps = timesteps.to(noisy_samples.device)
        shape = (-1,) + (1,) * (noisy_samples.dim() - 1)
        sa = (ac[timesteps] ** 0.5).flatten().view(shape)
        sb = ((1 - ac[timesteps]) ** 0.5).flatten().view(shape)
        return (noisy_samples - sb * noise) / (sa * scale)

    def __str__(self) -> str:
        return (f"DDIMScheduler(num_inference_steps={self.num_inference_steps}, "
                f"num_train_timesteps={self.num_train_timesteps}, prediction_type={self.prediction_type}, "
                f"beta_start={self.beta_start}, beta_end={self.beta_end}, beta_schedule={self.beta_schedule}, "
                f"clip_sample={self.clip_sample}, steps_offset={self.steps_offset}, weight_mode={self.weight_mode})")

    __repr__ = __str__

    def __len__(self) -> int:
        return self.num_train_timesteps
