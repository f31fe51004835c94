"""DPM-Solver++ multistep sampler: the schedule against the oracle restatement (oracle/dpm_solver_oracle.py), the math
of the solver on its own (order 1 is DDIM; order 2 converges faster on Gaussian data), and on the GPU the fused
ldm_dpmpp_step kernel, sample() and compute_pq with the scheduler.

Stated tolerances:
  schedule, scalar table, fused update : bit-exact (fp32)
  order-1 update vs DDIM (float64)     : 1e-12 absolute
  sample(), T DPM steps vs oracle      : relative L2 <= 8e-2 on the final latents (as the DDIM sampler test)
"""
import numpy as np
import pytest
import torch

from oracle import dpm_solver_oracle as DO
from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.schedulers import DPMSolverMultistepScheduler

KW = dict(num_train_timesteps=1000, beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear")
DEV = "cuda"


def _bits(t):
    return t.to(torch.float32).contiguous().view(torch.int32)


# ---------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("N", [1, 2, 10, 15, 50])
@pytest.mark.parametrize("schedule,order", [("scaled_linear", 2), ("linear", 2), ("scaled_linear", 1)])
def test_timesteps_and_scalar_table_match_oracle(N, schedule, order):
    kw = {**KW, "beta_schedule": schedule}
    s = DPMSolverMultistepScheduler(**kw, solver_order=order)
    s.set_timesteps(N)
    o = DO.DPMSolverOracle(**kw, solver_order=order)
    o.set_timesteps(N)
    assert s.timesteps.dtype == torch.int64 and torch.equal(s.timesteps, o.timesteps)
    assert torch.equal(_bits(s.sigmas), _bits(o.sigmas))
    tab = s.step_coefficients()
    assert tab.shape == (N, 8) and tab.dtype == torch.float32
    for i in range(N):
        o.lower_order_nums = min(i, order)     # the oracle's state after i steps of a trajectory
        k_order = o.order_of(i)
        k = o.scalars(i, k_order)
        assert float(tab[i, 6]) == k_order, i
        want = [k["sig"], k["alpha"], k["A"], k["Bc"]] + ([k["c"], k["hb"]] if k_order == 2 else [])
        assert torch.equal(_bits(tab[i, :len(want)]), _bits(torch.stack(want))), i
    if N > 2 and order == 2:
        assert (tab[1:-1, 6] == 2).all() and tab[0, 6] == 1 and tab[-1, 6] == 1
    # the last step goes to sigma = 0: prev is x0 (A = 0, Bc = -1)
    assert tab[-1, 2] == 0 and tab[-1, 3] == -1


@pytest.mark.parametrize("option", [
    {"beta_schedule": "squaredcos_cap_v2"}, {"solver_order": 3}, {"prediction_type": "v_prediction"},
    {"algorithm_type": "sde-dpmsolver++"}, {"algorithm_type": "dpmsolver"}, {"solver_type": "heun"},
    {"timestep_spacing": "leading"}, {"final_sigmas_type": "sigma_min"}, {"lower_order_final": False},
    {"use_karras_sigmas": True}, {"thresholding": True}, {"euler_at_final": True}, {"trained_betas": [0.1] * 1000},
    {"use_lu_lambdas": True}, {"variance_type": "learned_range"}, {"lambda_min_clipped": -5.1},
])
def test_options_outside_the_built_scope_raise(option):
    name = next(iter(option))
    with pytest.raises(NotImplementedError, match=name):
        DPMSolverMultistepScheduler(**{**KW, **option})


def test_scheduler_rejects_cpu_tensors_and_an_unset_schedule():
    from video_latent_diffusion_panoptic_segmentation_b200 import _lib as L
    s = DPMSolverMultistepScheduler(**KW)
    with pytest.raises(L.LdmError):
        s.coef_table("cpu")
    s.set_timesteps(10)
    assert s.init_noise_sigma == 1.0 and s.timesteps.numel() == 10
    with pytest.raises(L.LdmError):
        s.step(torch.zeros(4), int(s.timesteps[0]), torch.zeros(4))   # CPU tensors: no fallback


@pytest.mark.parametrize("N", [10, 50])
def test_first_order_update_is_ddim_in_float64(N):
    """With alpha = sqrt(abar), sig = sqrt(1 - abar), the first-order update reduces to alpha_t x0 + sig_t eps: DDIM from
    t_i to t_{i+1} (abar = 1 after the last step)."""
    o = DO.DPMSolverOracle(**KW, solver_order=1, dtype=torch.float64)
    o.set_timesteps(N)
    ac = o.alphas_cumprod
    g = torch.Generator().manual_seed(3)
    x = torch.randn(4096, generator=g, dtype=torch.float64)
    ts = o.timesteps.tolist()
    for i, t in enumerate(ts):
        eps = torch.randn(4096, generator=g, dtype=torch.float64)
        a_t = ac[t]
        a_p = ac[ts[i + 1]] if i + 1 < N else torch.tensor(1.0, dtype=torch.float64)
        x0 = (x - (1 - a_t) ** 0.5 * eps) / a_t ** 0.5
        ddim = a_p ** 0.5 * x0 + (1 - a_p) ** 0.5 * eps
        prev, _ = o.step(eps, t, x)
        assert (prev - ddim).abs().max().item() <= 1e-12, i
        x = prev


@pytest.mark.parametrize("N", [10, 20])
def test_second_order_is_closer_to_the_exact_flow_on_gaussian_data(N):
    """Data N(0, s^2), s^2 = 0.25: the exact noise prediction is eps = sig x / (alpha^2 s^2 + sig^2) and the probability
    flow maps x_T to x_T std(sigma_k) / std(sigma_0), std^2 = alpha^2 s^2 + sig^2. Stopping before the final sigma = 0
    step, the second-order state is at least 5x closer to it than the first-order state (float64)."""
    s2 = 0.25
    err = {}
    for order in (1, 2):
        o = DO.DPMSolverOracle(**KW, solver_order=order, dtype=torch.float64)
        o.set_timesteps(N)

        def std(k):
            a, sg, _ = o.alpha_sigma_lambda(k)
            return (a * a * s2 + sg * sg).sqrt()
        xT = torch.randn(100000, generator=torch.Generator().manual_seed(0), dtype=torch.float64) * std(0)
        x = xT.clone()
        for i in range(N - 1):
            a, sg, _ = o.alpha_sigma_lambda(i)
            x, _ = o.step(sg * x / (a * a * s2 + sg * sg), o.timesteps[i], x)
        exact = xT * std(N - 1) / std(0)
        err[order] = ((x - exact).norm() / exact.norm()).item()
    assert err[2] * 5 <= err[1], err


# ---------------------------------------------------------------------------------------------------------- GPU
def _rel(got, ref):
    got, ref = got.float(), ref.float()
    return ((got - ref).pow(2).sum().sqrt() / (ref.pow(2).sum().sqrt() + 1e-12)).item()


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(2, 4, 6, 10), (3, 1, 7, 11)], ids=["n%4=0", "tail"])
@pytest.mark.parametrize("inplace", [False, True])
@pytest.mark.parametrize("cfg", [False, True])
def test_kernel_matches_oracle_bit_for_bit_over_a_trajectory(shape, inplace, cfg):
    from video_latent_diffusion_panoptic_segmentation_b200 import ops
    N, g = 12, 7.5
    s = DPMSolverMultistepScheduler(**KW)
    s.set_timesteps(N)
    o = DO.DPMSolverOracle(**KW)
    o.set_timesteps(N)
    gen = torch.Generator().manual_seed(5)
    x_ref = torch.randn(shape, generator=gen)
    eps_seq = [(torch.randn(shape, generator=gen), torch.randn(shape, generator=gen)) for _ in range(N)]
    coef, steps = s.coef_table(DEV), s.step_index_table(DEV)
    x = x_ref.to(DEV)
    x0_prev = torch.empty_like(x)
    for i, t in enumerate(s.timesteps.tolist()):
        u, tx = eps_seq[i]
        eps = u + g * (tx - u) if cfg else u
        prev_ref, x0_ref = o.step(eps, t, x_ref)
        prev = x if inplace else torch.empty_like(x)
        ops.dpmpp_step(u.to(DEV), x, coef, steps[i:i + 1], prev, x0_prev,
                       eps_text=tx.to(DEV) if cfg else None, guidance_scale=g if cfg else 0.0)
        assert torch.equal(_bits(prev.cpu()), _bits(prev_ref)), i
        assert torch.equal(_bits(x0_prev.cpu()), _bits(x0_ref)), i
        x, x_ref = prev, prev_ref


@pytest.mark.gpu
def test_scheduler_step_is_stateful_and_bit_exact():
    """step(model_output, t, sample) -> prev_sample, the diffusers contract: the scheduler carries the previous x0."""
    N, shape = 8, (2, 4, 5, 9)
    s = DPMSolverMultistepScheduler(**KW)
    s.set_timesteps(N, device=DEV)
    o = DO.DPMSolverOracle(**KW)
    o.set_timesteps(N)
    gen = torch.Generator().manual_seed(11)
    x_ref = torch.randn(shape, generator=gen)
    x = x_ref.to(DEV)
    for t in s.timesteps:
        eps = torch.randn(shape, generator=gen)
        x = s.step(eps.to(DEV), t, x).prev_sample
        x_ref, _ = o.step(eps, int(t), x_ref)
        assert torch.equal(_bits(x.cpu()), _bits(x_ref))
    assert s.step_index == N
    s.set_timesteps(N, device=DEV)          # a new trajectory
    with pytest.raises(NotImplementedError):
        s.step(x, s.timesteps[3], x)        # that does not start at timesteps[0]


@pytest.fixture(scope="module")
def models():
    from oracle import unet_oracle as UO
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.models import GeneralVAESeg, UNet, unet_init
    o_unet = UO.build_unet(seed=0)
    unet = UNet(device=DEV)
    unet.load_state_dict(o_unet.state_dict())
    unet.remove_cross_attention()
    kw = dict(in_channels=16, int_channels=256, out_channels=128, latent_channels=4, num_upscalers=2,
              upscale_channels=256, norm_num_groups=32, scaling_factor=0.2)
    vae = GeneralVAESeg(**kw, device=DEV)
    vae.load_state_dict(unet_init.random_seg_decoder_state_dict(seed=1, **kw))
    return dict(o_unet=o_unet.to(DEV), unet=unet, vae=vae)


def _rgb(B, h, w):
    return (0.18215 * torch.randn((B, 4, h, w), generator=torch.Generator().manual_seed(1234))).to(DEV)


@pytest.mark.gpu
def test_sampler_vs_oracle(models):
    from oracle import ldmseg_oracle as LO
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.trainers import TrainerDiffusion
    B, h, w, T = 2, 16, 24, 5
    rgb = _rgb(B, h, w)
    tr = TrainerDiffusion(p={}, vae_semseg=models["vae"], unet_model=models["unet"],
                          noise_scheduler=DPMSolverMultistepScheduler(**KW), args={"gpu": 0})
    lat = tr.sample([""] * B, num_inference_steps=T, seed=42, rgb_latents=rgb)
    ref = LO.sample(models["o_unet"], DO.DPMSolverOracle(**KW), rgb, num_inference_steps=T, seed=42)
    assert lat.shape == ref.shape == (B, 4, h, w)
    assert _rel(lat, ref) < 8e-2, _rel(lat, ref)
    # the solver order matters more than the error
    ref1 = LO.sample(models["o_unet"], DO.DPMSolverOracle(**KW, solver_order=1), rgb, num_inference_steps=T, seed=42)
    assert _rel(ref1, ref) > _rel(lat, ref)
    # return_all_latents: one state per step, the last is the result
    allv = tr.sample([""] * B, num_inference_steps=T, seed=42, rgb_latents=rgb, return_all_latents=True)
    assert allv.shape == (T * B, 4, h, w) and torch.equal(allv[-B:], lat)


@pytest.mark.gpu
def test_graph_replay_equals_eager_and_runs_are_bit_identical(models):
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.trainers import TrainerDiffusion
    B, h, w, T = 2, 16, 24, 6
    rgb = _rgb(B, h, w)
    sched = DPMSolverMultistepScheduler(**KW)
    tr = TrainerDiffusion(p={}, unet_model=models["unet"], noise_scheduler=sched, args={"gpu": 0})
    lat = tr.sample([""] * B, num_inference_steps=T, seed=7, rgb_latents=rgb)
    lat2 = tr.sample([""] * B, num_inference_steps=T, seed=7, rgb_latents=rgb)
    assert torch.equal(lat, lat2)
    plan = tr._loop_state(B, h, w)["plan"]
    assert plan.graph is not None
    graph, plan.graph = plan.graph, None     # the same plan, run eagerly launch by launch
    try:
        lat_eager = tr.sample([""] * B, num_inference_steps=T, seed=7, rgb_latents=rgb)
    finally:
        plan.graph = graph
    assert torch.equal(lat, lat_eager)


@pytest.mark.gpu
def test_sampler_classifier_free_guidance_vs_oracle():
    from types import SimpleNamespace
    from oracle import ldmseg_oracle as LO
    from oracle import unet_oracle as UO
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.models import UNet
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.trainers import TrainerDiffusion

    class Tok:
        model_max_length = 12

        def __call__(self, texts, padding="max_length", max_length=None, truncation=True, return_tensors="pt"):
            L_ = max_length or self.model_max_length
            ids = torch.zeros((len(texts), L_), dtype=torch.long)
            for i, t in enumerate(texts):
                codes = [1 + (ord(c) % 60) for c in t][:L_]
                ids[i, :len(codes)] = torch.tensor(codes, dtype=torch.long)
            return SimpleNamespace(input_ids=ids)

    class Enc(torch.nn.Module):
        def __init__(self):
            super().__init__()
            torch.manual_seed(12)
            self.emb = torch.nn.Embedding(64, 768)
            self.pos = torch.nn.Parameter(0.1 * torch.randn(12, 768))

        def forward(self, input_ids):
            return (self.emb(input_ids) + self.pos[None, :input_ids.shape[1]],)

    o_unet = UO.build_unet(seed=8, cross_attention_dim=768)
    unet = UNet(device=DEV)
    unet.load_state_dict(o_unet.state_dict())
    o_unet = o_unet.to(DEV)
    tok, enc = Tok(), Enc().to(DEV).eval()
    B, h, w, T, g = 2, 16, 24, 4, 4.0
    prompts = ["a car on the road", "two pedestrians"]
    rgb = _rgb(B, h, w)
    sched = DPMSolverMultistepScheduler(**KW)
    sched.set_timesteps(T)
    tr = TrainerDiffusion(p={}, unet_model=unet, tokenizer=tok, text_encoder=enc, args={"gpu": 0})
    lat = tr.sample(prompts, num_inference_steps=T, guidance_scale=g, seed=42, rgb_latents=rgb, scheduler=sched)
    with torch.no_grad():
        ctx = enc(tok(prompts).input_ids.to(DEV))[0]
        unc = enc(tok([""] * B).input_ids.to(DEV))[0]
    ref = LO.sample(o_unet, DO.DPMSolverOracle(**KW), rgb, num_inference_steps=T, seed=42, context=ctx,
                    uncond_context=unc, guidance_scale=g)
    ref1 = LO.sample(o_unet, DO.DPMSolverOracle(**KW), rgb, num_inference_steps=T, seed=42, context=ctx,
                     uncond_context=unc, guidance_scale=1.0)
    assert lat.shape == ref.shape == (B, 4, h, w)
    assert _rel(lat, ref) < 8e-2, _rel(lat, ref)
    assert _rel(ref1, ref) > 2 * _rel(lat, ref)  # the guidance scale matters more than the error


@pytest.mark.gpu
def test_sampler_rejects_self_condition_and_foreign_schedulers(models):
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.trainers import TrainerDiffusion
    rgb = _rgb(1, 16, 24)
    tr = TrainerDiffusion(p={"train_kwargs": {"self_condition": True}}, unet_model=models["unet"],
                          noise_scheduler=DPMSolverMultistepScheduler(**KW), args={"gpu": 0})
    with pytest.raises(NotImplementedError, match="self_condition"):
        tr.sample([""], num_inference_steps=4, seed=0, rgb_latents=rgb)

    class Foreign:
        timesteps = torch.arange(3)
        init_noise_sigma = 1.0

        def step(self, *a, **k):
            raise AssertionError("not reached")

    tr = TrainerDiffusion(p={}, unet_model=models["unet"], args={"gpu": 0})
    with pytest.raises(NotImplementedError, match="Foreign"):
        tr.sample([""], num_inference_steps=3, seed=0, rgb_latents=rgb, scheduler=Foreign())


@pytest.mark.gpu
def test_compute_pq_with_dpm_scheduler(models):
    from oracle import eval_oracle as EO
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.trainers import TrainerDiffusion
    B, h, w, T = 2, 16, 24, 4
    H, W = 8 * h, 8 * w
    rng = np.random.default_rng(7)
    batches = []
    for i in range(2):
        rgb = 0.18215 * torch.randn((B, 4, h, w), generator=torch.Generator().manual_seed(1234 + i))
        gt = torch.from_numpy(rng.integers(0, 19, size=(B, H, W)).astype(np.int64))
        batches.append({"rgb_latents": rgb, "semseg": gt})
    p = {"eval_kwargs": {"mask_th": 0.0, "count_th": 64, "overlap_th": 0.0}, "ignore_label": 127}
    tr = TrainerDiffusion(p=p, vae_semseg=models["vae"], unet_model=models["unet"],
                          noise_scheduler=DPMSolverMultistepScheduler(**KW), args={"gpu": 0})
    res = tr.compute_metrics(["pq"], seed=42, dataloader=batches, num_inference_steps=T)
    assert tr.noise_scheduler.timesteps.numel() == T
    ev = EO.CityscapesPQOracle()
    for data, cleaned in zip(batches, tr.last_cleaned):
        for b in range(B):
            ev.add_image(cleaned[b].cpu().numpy().astype(np.int64), data["semseg"][b].numpy())
    want = ev.evaluate()
    for k in ("pq", "sq", "rq", "tp", "fp", "fn", "iou_sum"):
        assert res[k] == want[k], k
