"""ORACLE (test infrastructure only): CPU restatement of DPM-Solver++ multistep sampling (Lu et al. 2022,
arXiv:2211.01095) in the form diffusers' ``DPMSolverMultistepScheduler`` runs it with algorithm_type="dpmsolver++",
solver_type="midpoint", prediction_type="epsilon", timestep_spacing="linspace", final_sigmas_type="zero",
lower_order_final=True and solver_order 1 or 2.

Written from the formulas, not from the mirror: a stateful scheduler with the list of previous x0 predictions
(``model_outputs``), as diffusers keeps it. ``dtype=torch.float32`` keeps every scalar and element-wise op in fp32 (the
mirror's kernel is bit-exact with it); ``dtype=torch.float64`` runs the schedule and the steps in float64 (the math
checks: the order-1 / DDIM identity, convergence order on Gaussian data).

The step returns (prev_sample, x0) so ``ldmseg_oracle.sample`` drives it as it drives DDIMOracle; the last step goes
to sigma = 0, where prev_sample equals x0.
"""
import numpy as np
import torch


class DPMSolverOracle:
    def __init__(self, num_train_timesteps=1000, beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear",
                 solver_order=2, dtype=torch.float32, **unused):
        if beta_schedule == "scaled_linear":
            betas = torch.linspace(beta_start ** 0.5, beta_end ** 0.5, num_train_timesteps, dtype=dtype) ** 2
        elif beta_schedule == "linear":
            betas = torch.linspace(beta_start, beta_end, num_train_timesteps, dtype=dtype)
        else:
            raise NotImplementedError(beta_schedule)
        assert solver_order in (1, 2)
        self.dtype = dtype
        self.alphas_cumprod = torch.cumprod(1.0 - betas, dim=0)
        self.num_train_timesteps = num_train_timesteps
        self.solver_order = solver_order
        self.init_noise_sigma = 1.0
        self.num_inference_steps = None

    def set_timesteps(self, num_inference_steps):
        T, N = self.num_train_timesteps, num_inference_steps
        self.num_inference_steps = N
        ts = np.linspace(0, T - 1, N + 1).round()[::-1][:-1].copy().astype(np.int64)
        self.timesteps = torch.from_numpy(ts)
        sigmas = ((1 - self.alphas_cumprod) / self.alphas_cumprod) ** 0.5
        sigmas = sigmas[self.timesteps]
        self.sigmas = torch.cat([sigmas, torch.zeros(1, dtype=self.dtype)]).to(self.dtype)
        self.model_outputs = [None] * self.solver_order
        self.lower_order_nums = 0
        self.step_index = None

    set_timesteps_inference = set_timesteps

    def alpha_sigma_lambda(self, k):
        """(alpha, sig, lam) of sigma_k, 0-dim tensors of self.dtype."""
        s = self.sigmas[k]
        alpha = 1 / ((s ** 2 + 1) ** 0.5)
        sig = s * alpha
        return alpha, sig, torch.log(alpha) - torch.log(sig)

    def scalars(self, i, order):
        """The scalars of step i: sig_i, alpha_i, A, Bc and, at order 2, c = 1 / r0 and 0.5 * Bc."""
        alpha_s, sig_s, lam_s = self.alpha_sigma_lambda(i)
        alpha_t, sig_t, lam_t = self.alpha_sigma_lambda(i + 1)
        h = lam_t - lam_s
        out = {"sig": sig_s, "alpha": alpha_s, "A": sig_t / sig_s, "Bc": alpha_t * (torch.exp(-h) - 1.0)}
        if order == 2:
            _, _, lam_s1 = self.alpha_sigma_lambda(i - 1)
            r0 = (lam_s - lam_s1) / h
            out["c"] = 1.0 / r0
            out["hb"] = 0.5 * out["Bc"]
        return out

    def order_of(self, i):
        last = i == self.num_inference_steps - 1   # final_sigmas_type="zero" forces first order there
        return 1 if (self.solver_order == 1 or self.lower_order_nums < 1 or last) else 2

    def step(self, model_output, timestep, sample):
        if self.step_index is None:
            self.step_index = int((self.timesteps == int(timestep)).nonzero()[0])
        i = self.step_index
        order = self.order_of(i)
        k = self.scalars(i, order)
        x0 = (sample - k["sig"] * model_output) / k["alpha"]
        self.model_outputs = self.model_outputs[1:] + [x0]
        if order == 1:
            prev = k["A"] * sample - k["Bc"] * x0
        else:
            m0, m1 = self.model_outputs[-1], self.model_outputs[-2]
            D1 = k["c"] * (m0 - m1)
            prev = (k["A"] * sample - k["Bc"] * x0) - k["hb"] * D1
        if self.lower_order_nums < self.solver_order:
            self.lower_order_nums += 1
        self.step_index = i + 1
        return prev, x0
