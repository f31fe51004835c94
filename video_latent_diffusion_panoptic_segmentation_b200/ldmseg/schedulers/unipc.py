"""UniPC multistep sampler (Zhao et al. 2023, arXiv:2302.04867), as diffusers' ``UniPCMultistepScheduler`` runs it with
``predict_x0=True``, ``solver_type="bh2"``, epsilon prediction, ``timestep_spacing="linspace"``,
``final_sigmas_type="zero"`` and ``lower_order_final=True``, at solver order 1, 2 or 3 and with any
``disable_corrector`` list. Any other option raises.

Its predictor UniP is DPM-Solver++'s data-prediction update; its corrector UniC refines the result of the previous step
with the model output of the current one, which the step computes anyway, so it raises the order by one at no extra
UNet forward. ``solver_type="bh1"`` is not built: its B(h) = -h is infinite on the final step to sigma = 0.

Schedule (host, fp32): the betas, timesteps and sigmas of ``DPMSolverMultistepScheduler``, and per sigma
``alpha = 1 / (sigma**2 + 1) ** 0.5``, ``sig = sigma * alpha``, ``lam = log(alpha) - log(sig)``. An update from index a
to index t at order q has ``h = lam_t - lam_a``, ``hh = -h``, ``phi = B = expm1(hh)``, ``r_k = (lam_{a-k} - lam_a) / h``
(k = 1 .. q-1), and rho from R, b: with ``h_phi = phi / hh - 1`` and ``f = 1``, for j = 1 .. q row j-1 of R is
``(r_1 ** (j-1), .., r_{q-1} ** (j-1), 1)``, ``b_{j-1} = h_phi * f / B``, then ``f *= j + 1`` and
``h_phi = h_phi / hh - 1 / f``. The predictor of step i (a = i, t = i + 1) has order
``p_i = min(solver_order, N - i, i + 1)`` and ``rho = 0.5`` at p = 2, ``solve(R[:-1, :-1], b[:-1])`` at p = 3 (none at
p = 1). The corrector of step i > 0 (a = i - 1, t = i, order p_{i-1}) is skipped when i - 1 is in ``disable_corrector``;
its ``rho = 0.5`` at order 1, ``solve(R, b)`` otherwise.

Every scalar is built here with 0-dim fp32 tensor ops; one fused kernel (ldm_unipc_step) does the element-wise part —
guidance, the x0 prediction, the corrector, the predictor and the history shift — with round-to-nearest intrinsics in
the op order of oracle/unipc_oracle.py, so fp32 results are bit-identical to it. The kernel reads its row of the scalar
table by a device-side step index: the sampler loop needs no host sync. The last step goes to sigma = 0 at first order
(A = 0, Phi = -1): the result is the final x0 prediction exactly.
"""
from typing import Optional, Union

import numpy as np
import torch

from ..utils import OutputDict
from ... import _lib as L
from ... import ops
from .ddim_scheduler import make_betas

# sig_i, alpha_i, predictor order, corrector order (0: off); the predictor's A, Phi, Bh, r_1, r_2, rho_1, rho_2; the
# corrector's A, Phi, Bh, r_1, r_2, rho_1, rho_2, rho_m; 0 (include/ldmseg_b200.h, ldm_unipc_step)
COEF_COLS = 20


class UniPCMultistepSchedulerOutput(OutputDict):
    prev_sample: torch.Tensor


def _scope(name, value, allowed):
    if value not in allowed:
        raise NotImplementedError(f"UniPCMultistepScheduler: {name}={value!r} is not built (supported: "
                                  f"{', '.join(repr(a) for a in allowed)})")


class UniPCMultistepScheduler(object):
    order = 1  # diffusers' pipelines read it: one model call per step

    def __init__(self, num_train_timesteps: int = 1000, beta_start: float = 0.0001, beta_end: float = 0.02,
                 beta_schedule: str = "linear", trained_betas=None, solver_order: int = 2,
                 prediction_type: str = "epsilon", thresholding: bool = False, dynamic_thresholding_ratio: float = 0.995,
                 sample_max_value: float = 1.0, predict_x0: bool = True, solver_type: str = "bh2",
                 lower_order_final: bool = True, disable_corrector=(), solver_p=None,
                 use_karras_sigmas: bool = False, use_exponential_sigmas: bool = False, use_beta_sigmas: bool = False,
                 use_flow_sigmas: bool = False, flow_shift: float = 1.0, timestep_spacing: str = "linspace",
                 steps_offset: int = 0, final_sigmas_type: str = "zero", rescale_betas_zero_snr: bool = False):
        _scope("beta_schedule", beta_schedule, ("linear", "scaled_linear"))
        _scope("trained_betas", trained_betas, (None,))
        _scope("solver_order", solver_order, (1, 2, 3))
        _scope("prediction_type", prediction_type, ("epsilon",))
        _scope("thresholding", thresholding, (False,))
        _scope("predict_x0", predict_x0, (True,))
        _scope("solver_type", solver_type, ("bh2",))
        _scope("lower_order_final", lower_order_final, (True,))
        _scope("solver_p", solver_p, (None,))
        for name, v in (("use_karras_sigmas", use_karras_sigmas), ("use_exponential_sigmas", use_exponential_sigmas),
                        ("use_beta_sigmas", use_beta_sigmas), ("use_flow_sigmas", use_flow_sigmas),
                        ("rescale_betas_zero_snr", rescale_betas_zero_snr)):
            _scope(name, v, (False,))
        _scope("timestep_spacing", timestep_spacing, ("linspace",))
        _scope("final_sigmas_type", final_sigmas_type, ("zero",))
        self.betas = make_betas(beta_schedule, beta_start, beta_end, num_train_timesteps, owner=self.__class__)
        self.alphas = 1.0 - self.betas
        self.alphas_cumprod = torch.cumprod(self.alphas, dim=0)
        self.num_train_timesteps = num_train_timesteps
        self.beta_schedule, self.beta_start, self.beta_end = beta_schedule, beta_start, beta_end
        self.solver_order = solver_order
        self.prediction_type = prediction_type
        self.disable_corrector = [int(i) for i in disable_corrector]
        self.steps_offset = steps_offset  # unused with linspace spacing, as in diffusers
        self.init_noise_sigma = 1.0
        self.num_inference_steps = None
        self.timesteps = torch.from_numpy(np.arange(0, num_train_timesteps)[::-1].copy().astype(np.int64))
        self.sigmas = None
        self._table = None     # f32 [N, COEF_COLS] on the host
        self._coef_dev = {}    # device -> the table there
        self._steps_dev = {}   # device -> int32 [N] = 0 .. N-1, the step indices the kernel reads its row by
        self._step_index = None
        self._state = None     # [last, m1 .. m_order] of the trajectory step() is on

    # ------------------------------------------------------------------ schedule
    def set_timesteps(self, num_inference_steps: int, device: Union[str, torch.device] = None):
        if num_inference_steps < 1:
            raise L.LdmError(f"num_inference_steps must be at least 1, got {num_inference_steps}")
        T, N = self.num_train_timesteps, int(num_inference_steps)
        self.num_inference_steps = N
        ts = np.linspace(0, T - 1, N + 1).round()[::-1][:-1].copy().astype(np.int64)
        sig_all = ((1 - self.alphas_cumprod) / self.alphas_cumprod) ** 0.5
        self.sigmas = torch.cat([sig_all[torch.from_numpy(ts)], torch.zeros(1)]).to(torch.float32)
        self.timesteps = torch.from_numpy(ts).to(device)
        self._table = self.step_coefficients()
        self._coef_dev, self._steps_dev = {}, {}
        self._step_index, self._state = None, None

    def set_timesteps_inference(self, num_inference_steps: int, device: Union[str, torch.device] = None):
        """The name the trainer calls (TrainerDiffusion.sample / compute_pq)."""
        self.set_timesteps(num_inference_steps, device)

    def move_timesteps_to(self, device: Union[str, torch.device]):
        self.timesteps = self.timesteps.to(device)

    def predictor_order(self, i: int) -> int:
        """lower_order_final, and one more order per step until solver_order."""
        return min(self.solver_order, self.num_inference_steps - i, i + 1)

    def _update_scalars(self, lam, alpha, sig, a, t, q, corrector):
        """[A, Phi, Bh, r_1, r_2, rho_1, rho_2(, rho_m)] of the update a -> t at order q; unused entries are 0."""
        zero = torch.zeros((), dtype=torch.float32)
        h = lam[t] - lam[a]
        hh = -h
        phi = torch.expm1(hh)
        B = torch.expm1(hh)
        r = [(lam[a - k] - lam[a]) / h for k in range(1, q)]
        rho = []
        if corrector or q > 1:
            rks = torch.stack(r + [torch.ones((), dtype=torch.float32)])
            R, b = [], []
            h_phi, f = phi / hh - 1, 1
            for j in range(1, q + 1):
                R.append(torch.pow(rks, j - 1))
                b.append(h_phi * f / B)
                f *= j + 1
                h_phi = h_phi / hh - 1 / f
            R, b = torch.stack(R), torch.stack(b)
            half = torch.tensor([0.5], dtype=torch.float32)
            if corrector:
                rho = list(half if q == 1 else torch.linalg.solve(R, b))
            else:
                rho = list(half if q == 2 else torch.linalg.solve(R[:-1, :-1], b[:-1]))
        out = [sig[t] / sig[a], alpha[t] * phi, alpha[t] * B]
        out += r + [zero] * (2 - len(r))
        if corrector:   # the last rho weighs m - m1, the others the history differences
            out += rho[:-1] + [zero] * (3 - len(rho)) + [rho[-1]]
        else:
            out += rho + [zero] * (2 - len(rho))
        return out

    def step_coefficients(self) -> torch.Tensor:
        """f32 [N, COEF_COLS]: row i holds the scalars of step i, each a 0-dim fp32 tensor op in the order of the module
        docstring (the oracle, oracle/unipc_oracle.py, restates them independently)."""
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
            p = self.predictor_order(i)
            q = self.predictor_order(i - 1) if i > 0 and (i - 1) not in self.disable_corrector else 0
            pred = self._update_scalars(lam, alpha, sig, i, i + 1, p, corrector=False)
            corr = self._update_scalars(lam, alpha, sig, i - 1, i, q, corrector=True) if q else [zero] * 8
            rows.append(torch.stack([sig[i], alpha[i], torch.tensor(float(p)), torch.tensor(float(q))] + pred + corr
                                    + [zero]))
        return torch.stack(rows).to(torch.float32).contiguous()

    def coef_table(self, device) -> torch.Tensor:
        if self._table is None:
            raise L.LdmError("UniPCMultistepScheduler: call set_timesteps(num_inference_steps) first")
        device = torch.device(device)
        if device not in self._coef_dev:
            self._coef_dev[device] = self._table.to(device)
        return self._coef_dev[device]

    def step_index_table(self, device) -> torch.Tensor:
        """int32 [N] = 0 .. N-1 on `device`: element i is the device-side index ldm_unipc_step reads row i by."""
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
            raise L.LdmError(f"UniPCMultistepScheduler.step: timestep {t} is not in the schedule")
        return hits[0]

    def step(self, model_output: torch.Tensor, timestep, sample: torch.Tensor,
             return_dict: bool = True) -> UniPCMultistepSchedulerOutput:
        """One corrector + predictor step, from the sample at `timestep` to the next one. The scheduler keeps the step
        index, the corrected sample of the previous step and the previous x0 predictions between calls, as diffusers'
        does; set_timesteps starts a new trajectory, which has to begin at timesteps[0]. The timestep is read once, at
        the first call."""
        if not (model_output.is_cuda and sample.is_cuda):
            raise L.LdmError("UniPCMultistepScheduler.step needs CUDA tensors: there is no CPU fallback")
        if self._table is None:
            raise L.LdmError("UniPCMultistepScheduler: call set_timesteps(num_inference_steps) first")
        if self._step_index is None:
            i = self._index_for_timestep(timestep)
            if i != 0:
                raise NotImplementedError("UniPCMultistepScheduler.step: a trajectory that starts after "
                                          "timesteps[0] is not built")
            self._step_index = 0
        i = self._step_index
        if i >= self.num_inference_steps:
            raise L.LdmError("UniPCMultistepScheduler.step: the schedule is exhausted; call set_timesteps again")
        dev = sample.device
        eps = model_output.contiguous().float()
        x = sample.contiguous().float()
        if self._state is None:
            self._state = [torch.empty_like(x) for _ in range(1 + self.solver_order)]
        elif self._state[0].shape != x.shape or self._state[0].device != dev:
            raise L.LdmError(f"UniPCMultistepScheduler.step: sample {tuple(x.shape)} on {dev} does not continue the "
                             f"trajectory of {tuple(self._state[0].shape)} on {self._state[0].device}")
        prev = torch.empty_like(x)
        ops.unipc_step(eps, x, self.coef_table(dev), self.step_index_table(dev)[i:i + 1], prev, self._state[0],
                       self._state[1:])
        self._step_index = i + 1
        if not return_dict:
            return (prev,)
        return UniPCMultistepSchedulerOutput(prev_sample=prev)

    def __str__(self) -> str:
        return (f"UniPCMultistepScheduler(num_inference_steps={self.num_inference_steps}, "
                f"num_train_timesteps={self.num_train_timesteps}, solver_order={self.solver_order}, "
                f"disable_corrector={self.disable_corrector}, beta_start={self.beta_start}, "
                f"beta_end={self.beta_end}, beta_schedule={self.beta_schedule})")

    __repr__ = __str__

    def __len__(self) -> int:
        return self.num_train_timesteps
