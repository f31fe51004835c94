"""DPM-Solver++ multistep sampler (Lu et al. 2022, arXiv:2211.01095), as diffusers' ``DPMSolverMultistepScheduler`` runs
it with ``algorithm_type="dpmsolver++"``, ``solver_type="midpoint"``, epsilon prediction, ``timestep_spacing="linspace"``,
``final_sigmas_type="zero"`` and ``lower_order_final=True``, at solver order 1 or 2. Any other option raises.

A second-order solver reaches DDIM-50 quality in 10-20 UNet forwards, and the forward is almost all of a sampler step.

Schedule (host, fp32, in this order): the betas of ``DDIMNoiseScheduler``; ``timesteps = linspace(0, T - 1, N + 1)
.round()[::-1][:-1]``; ``sigmas = ((1 - alphas_cumprod) / alphas_cumprod) ** 0.5`` at the timesteps, then a final 0;
per sigma ``alpha = 1 / (sigma**2 + 1) ** 0.5``, ``sig = sigma * alpha``, ``lam = log(alpha) - log(sig)``.
Step i (sigma_i -> sigma_{i+1}), with ``h = lam_{i+1} - lam_i``, ``A = sig_{i+1} / sig_i``,
``Bc = alpha_{i+1} * (exp(-h) - 1)``:
  x0   = (sample - sig_i * eps) / alpha_i
  prev = A * sample - Bc * x0                                  first order: order 1, i = 0 and the last step
  prev = (A * sample - Bc * x0) - (0.5 * Bc) * D1              second order, D1 = (1 / r0) * (x0 - x0_prev),
                                                               r0 = (lam_i - lam_{i-1}) / h
Every scalar is built here with 0-dim fp32 tensor ops; one fused kernel (ldm_dpmpp_step) does the element-wise part
with round-to-nearest intrinsics, so fp32 results are bit-identical to the same formulas in torch eager on the CPU.
The kernel reads its row of the scalar table by a device-side step index: the sampler loop needs no host sync.
"""
from typing import Optional, Union

import numpy as np
import torch

from ..utils import OutputDict
from ... import _lib as L
from ... import ops
from .ddim_scheduler import make_betas

COEF_COLS = 8  # sig_i, alpha_i, A, Bc, 1 / r0, 0.5 * Bc, order, 0 (include/ldmseg_b200.h, ldm_dpmpp_step)


class DPMSolverMultistepSchedulerOutput(OutputDict):
    prev_sample: torch.Tensor


def _scope(name, value, allowed):
    if value not in allowed:
        raise NotImplementedError(f"DPMSolverMultistepScheduler: {name}={value!r} is not built (supported: "
                                  f"{', '.join(repr(a) for a in allowed)})")


class DPMSolverMultistepScheduler(object):
    order = 1  # diffusers' pipelines read it: one model call per step

    def __init__(self, num_train_timesteps: int = 1000, beta_start: float = 0.0001, beta_end: float = 0.02,
                 beta_schedule: str = "linear", trained_betas=None, solver_order: int = 2,
                 prediction_type: str = "epsilon", thresholding: bool = False, dynamic_thresholding_ratio: float = 0.995,
                 sample_max_value: float = 1.0, algorithm_type: str = "dpmsolver++", solver_type: str = "midpoint",
                 lower_order_final: bool = True, euler_at_final: bool = False, use_karras_sigmas: bool = False,
                 use_exponential_sigmas: bool = False, use_beta_sigmas: bool = False, use_lu_lambdas: bool = False,
                 use_flow_sigmas: bool = False, flow_shift: float = 1.0, final_sigmas_type: str = "zero",
                 lambda_min_clipped: float = -float("inf"), variance_type: Optional[str] = None,
                 timestep_spacing: str = "linspace", steps_offset: int = 0, rescale_betas_zero_snr: bool = False):
        _scope("beta_schedule", beta_schedule, ("linear", "scaled_linear"))
        _scope("trained_betas", trained_betas, (None,))
        _scope("solver_order", solver_order, (1, 2))
        _scope("prediction_type", prediction_type, ("epsilon",))
        _scope("thresholding", thresholding, (False,))
        _scope("algorithm_type", algorithm_type, ("dpmsolver++",))
        _scope("solver_type", solver_type, ("midpoint",))
        _scope("lower_order_final", lower_order_final, (True,))
        _scope("euler_at_final", euler_at_final, (False,))
        for name, v in (("use_karras_sigmas", use_karras_sigmas), ("use_exponential_sigmas", use_exponential_sigmas),
                        ("use_beta_sigmas", use_beta_sigmas), ("use_lu_lambdas", use_lu_lambdas),
                        ("use_flow_sigmas", use_flow_sigmas), ("rescale_betas_zero_snr", rescale_betas_zero_snr)):
            _scope(name, v, (False,))
        _scope("final_sigmas_type", final_sigmas_type, ("zero",))
        _scope("lambda_min_clipped", lambda_min_clipped, (-float("inf"),))
        _scope("variance_type", variance_type, (None,))
        _scope("timestep_spacing", timestep_spacing, ("linspace",))
        self.betas = make_betas(beta_schedule, beta_start, beta_end, num_train_timesteps, owner=self.__class__)
        self.alphas = 1.0 - self.betas
        self.alphas_cumprod = torch.cumprod(self.alphas, dim=0)
        self.num_train_timesteps = num_train_timesteps
        self.beta_schedule, self.beta_start, self.beta_end = beta_schedule, beta_start, beta_end
        self.solver_order = solver_order
        self.prediction_type = prediction_type
        self.steps_offset = steps_offset  # unused with linspace spacing, as in diffusers
        self.init_noise_sigma = 1.0
        self.num_inference_steps = None
        self.timesteps = torch.from_numpy(np.arange(0, num_train_timesteps)[::-1].copy().astype(np.int64))
        self.sigmas = None
        self._table = None     # f32 [N, COEF_COLS] on the host
        self._coef_dev = {}    # device -> the table there
        self._steps_dev = {}   # device -> int32 [N] = 0 .. N-1, the step indices the kernel reads its row by
        self._step_index = None
        self._x0_prev = None

    # ------------------------------------------------------------------ schedule
    def set_timesteps(self, num_inference_steps: int, device: Union[str, torch.device] = None):
        if num_inference_steps < 1:
            raise L.LdmError(f"num_inference_steps must be at least 1, got {num_inference_steps}")
        T, N = self.num_train_timesteps, int(num_inference_steps)
        self.num_inference_steps = N
        ts = np.linspace(0, T - 1, N + 1).round()[::-1][:-1].copy().astype(np.int64)
        sig_all = ((1 - self.alphas_cumprod) / self.alphas_cumprod) ** 0.5
        sigmas = torch.cat([sig_all[torch.from_numpy(ts)], torch.zeros(1)]).to(torch.float32)
        self.sigmas = sigmas
        self.timesteps = torch.from_numpy(ts).to(device)
        self._table = self.step_coefficients()
        self._coef_dev, self._steps_dev = {}, {}
        self._step_index, self._x0_prev = None, None

    def set_timesteps_inference(self, num_inference_steps: int, device: Union[str, torch.device] = None):
        """The name the trainer calls (TrainerDiffusion.sample / compute_pq)."""
        self.set_timesteps(num_inference_steps, device)

    def move_timesteps_to(self, device: Union[str, torch.device]):
        self.timesteps = self.timesteps.to(device)

    def step_coefficients(self) -> torch.Tensor:
        """f32 [N, COEF_COLS]: row i holds the scalars of step i, each a 0-dim fp32 tensor op in the order of the module
        docstring (the oracle, oracle/dpm_solver_oracle.py, restates them independently)."""
        N = self.num_inference_steps
        alpha, sig, lam = [], [], []
        for s in self.sigmas:                 # 0-dim fp32 tensors
            a = 1 / ((s ** 2 + 1) ** 0.5)
            alpha.append(a)
            sig.append(s * a)
            lam.append(torch.log(a) - torch.log(s * a))
        zero = torch.zeros((), dtype=torch.float32)
        rows = []
        for i in range(N):
            h = lam[i + 1] - lam[i]
            A = sig[i + 1] / sig[i]
            Bc = alpha[i + 1] * (torch.exp(-h) - 1.0)
            second = self.solver_order == 2 and 0 < i < N - 1
            if second:
                r0 = (lam[i] - lam[i - 1]) / h
                c, hb = 1.0 / r0, 0.5 * Bc
            else:
                c, hb = zero, zero
            order = torch.tensor(2.0 if second else 1.0)
            rows.append(torch.stack([sig[i], alpha[i], A, Bc, c, hb, order, zero]))
        return torch.stack(rows).to(torch.float32).contiguous()

    def coef_table(self, device) -> torch.Tensor:
        if self._table is None:
            raise L.LdmError("DPMSolverMultistepScheduler: call set_timesteps(num_inference_steps) first")
        device = torch.device(device)
        if device not in self._coef_dev:
            self._coef_dev[device] = self._table.to(device)
        return self._coef_dev[device]

    def step_index_table(self, device) -> torch.Tensor:
        """int32 [N] = 0 .. N-1 on `device`: element i is the device-side index ldm_dpmpp_step reads row i by."""
        device = torch.device(device)
        if device not in self._steps_dev:
            self._steps_dev[device] = torch.arange(self.num_inference_steps, dtype=torch.int32, device=device)
        return self._steps_dev[device]

    # ------------------------------------------------------------------ stateful step (diffusers' contract)
    @property
    def step_index(self):
        return self._step_index

    def scale_model_input(self, sample: torch.Tensor, *args, **kwargs) -> torch.Tensor:
        return sample

    def _index_for_timestep(self, timestep) -> int:
        t = int(timestep.reshape(-1)[0].item()) if torch.is_tensor(timestep) else int(timestep)  # one sync per run
        hits = (self.timesteps.cpu() == t).nonzero().flatten().tolist()
        if not hits:
            raise L.LdmError(f"DPMSolverMultistepScheduler.step: timestep {t} is not in the schedule")
        return hits[0]

    def step(self, model_output: torch.Tensor, timestep, sample: torch.Tensor,
             return_dict: bool = True) -> DPMSolverMultistepSchedulerOutput:
        """One solver step, from the sample at `timestep` to the next one. The scheduler keeps the step index and the
        previous x0 prediction between calls, as diffusers' does; set_timesteps starts a new trajectory, which has to
        begin at timesteps[0]. The timestep is read once, at the first call."""
        if not (model_output.is_cuda and sample.is_cuda):
            raise L.LdmError("DPMSolverMultistepScheduler.step needs CUDA tensors: there is no CPU fallback")
        if self._table is None:
            raise L.LdmError("DPMSolverMultistepScheduler: call set_timesteps(num_inference_steps) first")
        if self._step_index is None:
            i = self._index_for_timestep(timestep)
            if i != 0:
                raise NotImplementedError("DPMSolverMultistepScheduler.step: a trajectory that starts after "
                                          "timesteps[0] is not built")
            self._step_index = 0
        i = self._step_index
        if i >= self.num_inference_steps:
            raise L.LdmError("DPMSolverMultistepScheduler.step: the schedule is exhausted; call set_timesteps again")
        dev = sample.device
        eps = model_output.contiguous().float()
        x = sample.contiguous().float()
        if self._x0_prev is None:
            self._x0_prev = torch.empty_like(x)
        elif self._x0_prev.shape != x.shape or self._x0_prev.device != dev:
            raise L.LdmError(f"DPMSolverMultistepScheduler.step: sample {tuple(x.shape)} on {dev} does not continue "
                             f"the trajectory of {tuple(self._x0_prev.shape)} on {self._x0_prev.device}")
        prev = torch.empty_like(x)
        ops.dpmpp_step(eps, x, self.coef_table(dev), self.step_index_table(dev)[i:i + 1], prev, self._x0_prev)
        self._step_index = i + 1
        if not return_dict:
            return (prev,)
        return DPMSolverMultistepSchedulerOutput(prev_sample=prev)

    def __str__(self) -> str:
        return (f"DPMSolverMultistepScheduler(num_inference_steps={self.num_inference_steps}, "
                f"num_train_timesteps={self.num_train_timesteps}, solver_order={self.solver_order}, "
                f"beta_start={self.beta_start}, beta_end={self.beta_end}, beta_schedule={self.beta_schedule})")

    __repr__ = __str__

    def __len__(self) -> int:
        return self.num_train_timesteps
