"""ORACLE (test infrastructure only): CPU restatement of UniPC multistep sampling (Zhao et al. 2023, arXiv:2302.04867)
in the form diffusers' ``UniPCMultistepScheduler`` runs it with predict_x0=True, solver_type="bh2",
prediction_type="epsilon", timestep_spacing="linspace", final_sigmas_type="zero", lower_order_final=True, solver_order
1, 2 or 3 and any ``disable_corrector`` list.

Written from the formulas, not from the mirror: a stateful scheduler with the list of previous x0 predictions
(``model_outputs``) and the sample the previous step started from after its correction (``last_sample``), as diffusers
keeps them. ``dtype=torch.float32`` keeps every scalar and element-wise op in fp32 (the mirror's kernel is bit-exact with
it); ``dtype=torch.float64`` runs the schedule and the steps in float64 (the math checks).

Schedule: the betas, timesteps and sigmas of DPM-Solver++ (oracle/dpm_solver_oracle.py), per sigma_k
alpha_k = 1 / sqrt(sigma_k^2 + 1), s_k = sigma_k alpha_k, lam_k = log(alpha_k) - log(s_k). An update from index a to
index t at order q has h = lam_t - lam_a, hh = -h, phi = B = expm1(hh), r_k = (lam_{a-k} - lam_a) / h (k = 1 .. q-1),
A = s_t / s_a, Phi = alpha_t * phi, Bh = alpha_t * B, and rho from R, b (see ``update_scalars``).

Element-wise op order of step i (the kernel, ldm_unipc_step, copies it; every line is separately rounded):
  eps  = u + g * (text - u)                                                          (classifier-free guidance only)
  m    = (x - s_i * eps) / alpha_i                                                   (x is the sample as passed in)
  corrector, a = i - 1, t = i, order q = p_{i-1}, skipped when i - 1 is in disable_corrector; m_1, m_2, m_3 are the
  x0 predictions of steps i-1, i-2, i-3:
    S    = rho_m * (m - m_1)                                                         (q = 1)
    S    = ((rho_1 * ((m_2 - m_1) / r_1)) [+ rho_2 * ((m_3 - m_1) / r_2)]) + rho_m * (m - m_1)   (q = 2 [3])
    x^c  = (A * last - Phi * m_1) - Bh * S                                           (x^c = x without a corrector)
  predictor, a = i, t = i + 1, order p_i = min(solver_order, N - i, i + 1):
    prev = A * x^c - Phi * m                                                         (p = 1: no sum, not a zero sum)
    prev = (A * x^c - Phi * m) - Bh * ((rho_1 * ((m_1 - m) / r_1)) [+ rho_2 * ((m_2 - m) / r_2)])   (p = 2 [3])
  then last <- x^c and the history shifts: m_3 <- m_2, m_2 <- m_1, m_1 <- m.
The last step goes to sigma = 0 at first order with A = 0 and Phi = -1, so prev equals m exactly.

The step returns (prev_sample, x0) so ``ldmseg_oracle.sample`` drives it as it drives DPMSolverOracle.
"""
import numpy as np
import torch


class UniPCOracle:
    def __init__(self, num_train_timesteps=1000, beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear",
                 solver_order=2, disable_corrector=(), dtype=torch.float32, **unused):
        if beta_schedule == "scaled_linear":
            betas = torch.linspace(beta_start ** 0.5, beta_end ** 0.5, num_train_timesteps, dtype=dtype) ** 2
        elif beta_schedule == "linear":
            betas = torch.linspace(beta_start, beta_end, num_train_timesteps, dtype=dtype)
        else:
            raise NotImplementedError(beta_schedule)
        assert solver_order in (1, 2, 3)
        self.dtype = dtype
        self.alphas_cumprod = torch.cumprod(1.0 - betas, dim=0)
        self.num_train_timesteps = num_train_timesteps
        self.solver_order = solver_order
        self.disable_corrector = list(disable_corrector)
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
        self.last_sample = None
        self.this_order = None
        self.step_index = None

    set_timesteps_inference = set_timesteps

    def alpha_sigma_lambda(self, k):
        """(alpha, sig, lam) of sigma_k, 0-dim tensors of self.dtype."""
        s = self.sigmas[k]
        alpha = 1 / ((s ** 2 + 1) ** 0.5)
        sig = s * alpha
        return alpha, sig, torch.log(alpha) - torch.log(sig)

    def order_of(self, i):
        """Predictor order of step i: lower_order_final, and a warm-up of one order per step."""
        return min(self.solver_order, self.num_inference_steps - i, i + 1)

    def update_scalars(self, a, t, q, corrector):
        """Scalars of the update from sigma_a to sigma_t at order q: A, Phi, Bh, r = [r_1 .. r_{q-1}] and rho (the
        predictor's q - 1 values, or the corrector's q values whose last one weighs m - m_1)."""
        alpha_a, sig_a, lam_a = self.alpha_sigma_lambda(a)
        alpha_t, sig_t, lam_t = self.alpha_sigma_lambda(t)
        h = lam_t - lam_a
        hh = -h
        phi = torch.expm1(hh)
        B = torch.expm1(hh)                                  # bh2
        r = [(self.alpha_sigma_lambda(a - k)[2] - lam_a) / h for k in range(1, q)]
        out = {"A": sig_t / sig_a, "Phi": alpha_t * phi, "Bh": alpha_t * B, "r": r, "rho": []}
        if not corrector and q == 1:
            return out                                       # the predictor's sum is left out
        rks = torch.stack(r + [torch.ones((), dtype=self.dtype)])
        R, b = [], []
        h_phi, f = phi / hh - 1, 1
        for j in range(1, q + 1):
            R.append(torch.pow(rks, j - 1))
            b.append(h_phi * f / B)
            f *= j + 1
            h_phi = h_phi / hh - 1 / f
        R, b = torch.stack(R), torch.stack(b)
        half = torch.tensor([0.5], dtype=self.dtype)
        if corrector:
            rho = half if q == 1 else torch.linalg.solve(R, b)
        else:
            rho = half if q == 2 else torch.linalg.solve(R[:-1, :-1], b[:-1])
        out["rho"] = list(rho)
        return out

    def step(self, model_output, timestep, sample):
        if self.step_index is None:
            self.step_index = int((self.timesteps == int(timestep)).nonzero()[0])
        i = self.step_index
        alpha_i, sig_i, _ = self.alpha_sigma_lambda(i)
        m = (sample - sig_i * model_output) / alpha_i
        hist = self.model_outputs[::-1]                      # hist[0] = m_1 (step i - 1), hist[1] = m_2, ...
        x = sample
        if i > 0 and (i - 1) not in self.disable_corrector:
            q = self.this_order
            k = self.update_scalars(i - 1, i, q, corrector=True)
            S = k["rho"][-1] * (m - hist[0])
            if q > 1:
                D = k["rho"][0] * ((hist[1] - hist[0]) / k["r"][0])
                for j in range(2, q):
                    D = D + k["rho"][j - 1] * ((hist[j] - hist[0]) / k["r"][j - 1])
                S = D + S
            x = (k["A"] * self.last_sample - k["Phi"] * hist[0]) - k["Bh"] * S
        self.model_outputs = self.model_outputs[1:] + [m]
        p = self.order_of(i)
        self.this_order = p
        self.last_sample = x
        k = self.update_scalars(i, i + 1, p, corrector=False)
        prev = k["A"] * x - k["Phi"] * m
        if p > 1:
            S = k["rho"][0] * ((hist[0] - m) / k["r"][0])
            for j in range(2, p):
                S = S + k["rho"][j - 1] * ((hist[j - 1] - m) / k["r"][j - 1])
            prev = prev - k["Bh"] * S
        self.step_index = i + 1
        return prev, m
