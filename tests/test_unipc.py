"""UniPC multistep sampler: the schedule against the oracle restatement (oracle/unipc_oracle.py), the math of the
solver on its own (identities with DDIM and DPM-Solver++ 2M, convergence on Gaussian data), and on the GPU the fused
ldm_unipc_step kernel, sample() and compute_pq with the scheduler.

Stated tolerances:
  schedule, scalar table, fused update      : bit-exact (fp32)
  order 1 / 2 without corrector (float64)   : 1e-12 absolute against DDIM / DPM-Solver++ 2M
  sample(), T UniPC steps vs oracle         : relative L2 <= 8e-2 on the final latents (as the DDIM sampler test)
"""
import math

import numpy as np
import pytest
import torch

from oracle import dpm_solver_oracle as DO
from oracle import unipc_oracle as UO
from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.schedulers import UniPCMultistepScheduler

KW = dict(num_train_timesteps=1000, beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear")
DEV = "cuda"


def _bits(t):
    return t.to(torch.float32).contiguous().view(torch.int32)


def _oracle_row(o, i):
    """Row i of the scalar table, from the oracle's own scalars (order of include/ldmseg_b200.h, ldm_unipc_step)."""
    z = torch.zeros((), dtype=torch.float32)
    p = o.order_of(i)
    q = o.order_of(i - 1) if i > 0 and (i - 1) not in o.disable_corrector else 0
    k = o.update_scalars(i, i + 1, p, corrector=False)
    pred = [k["A"], k["Phi"], k["Bh"]] + k["r"] + [z] * (2 - len(k["r"])) + k["rho"] + [z] * (2 - len(k["rho"]))
    if q:
        k = o.update_scalars(i - 1, i, q, corrector=True)
        corr = ([k["A"], k["Phi"], k["Bh"]] + k["r"] + [z] * (2 - len(k["r"])) + k["rho"][:-1]
                + [z] * (3 - len(k["rho"])) + [k["rho"][-1]])
    else:
        corr = [z] * 8
    alpha, sig, _ = o.alpha_sigma_lambda(i)
    return p, q, torch.stack([sig, alpha, torch.tensor(float(p)), torch.tensor(float(q))] + pred + corr + [z])


# ---------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("N", [1, 2, 3, 5, 10, 15, 50])
@pytest.mark.parametrize("order", [1, 2, 3])
@pytest.mark.parametrize("disable", [(), (0, 2, 3)], ids=["corrector", "some-disabled"])
@pytest.mark.parametrize("schedule", ["scaled_linear", "linear"])
def test_timesteps_and_scalar_table_match_oracle(N, order, disable, schedule):
    kw = {**KW, "beta_schedule": schedule}
    s = UniPCMultistepScheduler(**kw, solver_order=order, disable_corrector=list(disable))
    s.set_timesteps(N)
    o = UO.UniPCOracle(**kw, solver_order=order, disable_corrector=disable)
    o.set_timesteps(N)
    assert s.timesteps.dtype == torch.int64 and torch.equal(s.timesteps, o.timesteps)
    assert torch.equal(_bits(s.sigmas), _bits(o.sigmas))
    tab = s.step_coefficients()
    assert tab.shape == (N, 20) and tab.dtype == torch.float32
    assert torch.isfinite(tab).all()          # unused columns are 0, never inf or NaN
    for i in range(N):
        p, q, want = _oracle_row(o, i)
        assert p == min(order, N - i, i + 1) and (q == 0) == (i == 0 or i - 1 in disable), i
        assert torch.equal(_bits(tab[i]), _bits(want)), i
    # the last step goes to sigma = 0 at first order: prev = A * x - Phi * m is m, bit for bit
    assert tab[-1, 2] == 1 and tab[-1, 4] == 0 and tab[-1, 5] == -1
    g = torch.Generator().manual_seed(N)
    x, m = torch.randn(4096, generator=g), torch.randn(4096, generator=g)
    assert torch.equal(tab[-1, 4] * x - tab[-1, 5] * m, m)


@pytest.mark.parametrize("option", [
    {"beta_schedule": "squaredcos_cap_v2"}, {"solver_order": 4}, {"prediction_type": "v_prediction"},
    {"solver_type": "bh1"}, {"predict_x0": False}, {"solver_p": object()}, {"thresholding": True},
    {"timestep_spacing": "leading"}, {"timestep_spacing": "trailing"}, {"final_sigmas_type": "sigma_min"},
    {"lower_order_final": False}, {"use_karras_sigmas": True}, {"use_exponential_sigmas": True},
    {"use_beta_sigmas": True}, {"use_flow_sigmas": True}, {"trained_betas": [0.1] * 1000},
    {"rescale_betas_zero_snr": True},
])
def test_options_outside_the_built_scope_raise(option):
    name = next(iter(option))
    with pytest.raises(NotImplementedError, match=name):
        UniPCMultistepScheduler(**{**KW, **option})


def test_scheduler_rejects_cpu_tensors_and_an_unset_schedule():
    from video_latent_diffusion_panoptic_segmentation_b200 import _lib as L
    s = UniPCMultistepScheduler(**KW)
    with pytest.raises(L.LdmError):
        s.coef_table("cpu")
    s.set_timesteps(10)
    assert s.init_noise_sigma == 1.0 and s.timesteps.numel() == 10
    with pytest.raises(L.LdmError):
        s.step(torch.zeros(4), int(s.timesteps[0]), torch.zeros(4))   # CPU tensors: no fallback


@pytest.mark.parametrize("N", [10, 50])
def test_first_order_without_corrector_is_ddim_in_float64(N):
    """UniP-1 is the first-order DPM-Solver++ update, alpha_t x0 + sig_t eps: DDIM from t_i to t_{i+1}."""
    o = UO.UniPCOracle(**KW, solver_order=1, disable_corrector=range(N), dtype=torch.float64)
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


@pytest.mark.parametrize("N", [5, 10, 50])
def test_second_order_without_corrector_is_dpm_solver_2m_in_float64(N):
    """UniP-2 with rho = 0.5 and B(h) = expm1(-h) is the midpoint DPM-Solver++ update: r_1 = -r0 and
    D_1 = (m_{i-1} - m_i) / r_1 = (m_i - m_{i-1}) / r0."""
    u = UO.UniPCOracle(**KW, solver_order=2, disable_corrector=range(N), dtype=torch.float64)
    u.set_timesteps(N)
    d = DO.DPMSolverOracle(**KW, solver_order=2, dtype=torch.float64)
    d.set_timesteps(N)
    g = torch.Generator().manual_seed(3)
    x = y = torch.randn(4096, generator=g, dtype=torch.float64)
    for i, t in enumerate(u.timesteps.tolist()):
        eps = torch.randn(4096, generator=g, dtype=torch.float64)
        x, _ = u.step(eps, t, x)
        y, _ = d.step(eps, t, y)
        assert (x - y).abs().max().item() <= 1e-12, i


S2 = 0.25   # data N(0, S2): eps(x) = sig x / (alpha^2 S2 + sig^2), and the flow scales x by std(sigma) / std(sigma_0)


def _gaussian_flow_error(o, N):
    """Relative distance to the exact flow of the state after N - 1 steps, the sample the last UNet forward sees (the
    last step, to sigma = 0, returns that forward's x0 prediction)."""
    def std(k):
        a, sg, _ = o.alpha_sigma_lambda(k)
        return (a * a * S2 + sg * sg).sqrt()
    xT = torch.randn(100000, generator=torch.Generator().manual_seed(0), dtype=torch.float64) * std(0)
    x = xT.clone()
    for i in range(N - 1):
        a, sg, _ = o.alpha_sigma_lambda(i)
        x, _ = o.step(sg * x / (a * a * S2 + sg * sg), o.timesteps[i], x)
    exact = xT * std(N - 1) / std(0)
    return ((x - exact).norm() / exact.norm()).item()


def test_unipc2_is_closer_to_the_exact_flow_than_dpm_solver_2m_at_10_steps():
    """On the Gaussian-data flow of test_dpm_solver.py (linspace timesteps), in float64: at N = 10 UniPC-2 ends 31.8x
    closer than DPM-Solver++ 2M (2.2e-4 against 7.1e-3). The ordering is not monotone in N on this schedule: at N = 20
    UniPC-2 ends farther (4.3e-3 against 3.2e-3), and UniPC-3 ends farther than UniPC-2 at N = 10 (1.2e-3) and 20
    (4.4e-3). Those are not asserted; the convergence orders are, on a geometric grid, below."""
    N = 10
    u = UO.UniPCOracle(**KW, solver_order=2, dtype=torch.float64)
    u.set_timesteps(N)
    d = DO.DPMSolverOracle(**KW, solver_order=2, dtype=torch.float64)
    d.set_timesteps(N)
    err_u, err_d = _gaussian_flow_error(u, N), _gaussian_flow_error(d, N)
    assert err_u * 30 <= err_d, (err_u, err_d)


def test_convergence_orders_on_a_geometric_sigma_grid():
    """Sigmas log-spaced from 10 to 0.3 (then the final 0), the Gaussian-data flow in float64: UniPC at solver order p
    converges at order p + 1 (the corrector adds one). Measured error ratios from N = 41 to 81 (the step halves):
    DPM-Solver++ 2M 4.7, UniPC-1 4.0, UniPC-2 7.5, UniPC-3 8.0 (lower_order_final caps it at three); UniPC-2 is 2.5x to
    5.2x closer than DPM-Solver++ 2M at N = 21, 41, 81."""
    def err(make, N):
        o = make()
        o.set_timesteps(N)
        o.sigmas = torch.cat([torch.exp(torch.linspace(math.log(10.0), math.log(0.3), N, dtype=torch.float64)),
                              torch.zeros(1, dtype=torch.float64)])
        return _gaussian_flow_error(o, N)
    arms = {"dpm2": lambda: DO.DPMSolverOracle(**KW, solver_order=2, dtype=torch.float64)}
    for p in (1, 2, 3):
        arms[f"unipc{p}"] = lambda p=p: UO.UniPCOracle(**KW, solver_order=p, dtype=torch.float64)
    e = {name: {N: err(make, N) for N in (21, 41, 81)} for name, make in arms.items()}
    ratio = {name: v[41] / v[81] for name, v in e.items()}
    assert ratio["unipc1"] >= 3.5 and ratio["unipc2"] >= 7.0 and ratio["unipc3"] >= 7.0, ratio
    for N in (21, 41, 81):
        assert e["unipc2"][N] * 2.5 <= e["dpm2"][N], (N, e)


# ---------------------------------------------------------------------------------------------------------- GPU
def _rel(got, ref):
    got, ref = got.float(), ref.float()
    return ((got - ref).pow(2).sum().sqrt() / (ref.pow(2).sum().sqrt() + 1e-12)).item()


@pytest.mark.gpu
@pytest.mark.parametrize("order", [1, 2, 3])
@pytest.mark.parametrize("shape", [(2, 4, 6, 10), (3, 1, 7, 11)], ids=["n%4=0", "tail"])
@pytest.mark.parametrize("inplace", [False, True])
@pytest.mark.parametrize("cfg", [False, True])
def test_kernel_matches_oracle_bit_for_bit_over_a_trajectory(order, shape, inplace, cfg):
    """Every output of every step: prev, the corrected sample and the newest x0. Without CFG the corrector runs at
    every step; with it, the corrector is disabled after steps 2 and 5."""
    from video_latent_diffusion_panoptic_segmentation_b200 import ops
    N, g = 12, 7.5
    disable = [2, 5] if cfg else []
    s = UniPCMultistepScheduler(**KW, solver_order=order, disable_corrector=disable)
    s.set_timesteps(N)
    o = UO.UniPCOracle(**KW, solver_order=order, disable_corrector=disable)
    o.set_timesteps(N)
    gen = torch.Generator().manual_seed(5)
    x_ref = torch.randn(shape, generator=gen)
    eps_seq = [(torch.randn(shape, generator=gen), torch.randn(shape, generator=gen)) for _ in range(N)]
    coef, steps = s.coef_table(DEV), s.step_index_table(DEV)
    x = x_ref.to(DEV)
    last = torch.empty_like(x)
    hist = [torch.empty_like(x) for _ in range(order)]
    for i, t in enumerate(s.timesteps.tolist()):
        u, tx = eps_seq[i]
        eps = u + g * (tx - u) if cfg else u
        prev_ref, x0_ref = o.step(eps, t, x_ref)
        prev = x if inplace else torch.empty_like(x)
        ops.unipc_step(u.to(DEV), x, coef, steps[i:i + 1], prev, last, hist,
                       eps_text=tx.to(DEV) if cfg else None, guidance_scale=g if cfg else 0.0)
        assert torch.equal(_bits(prev.cpu()), _bits(prev_ref)), i
        assert torch.equal(_bits(last.cpu()), _bits(o.last_sample)), i
        assert torch.equal(_bits(hist[0].cpu()), _bits(x0_ref)), i
        x, x_ref = prev, prev_ref
    assert torch.equal(x_ref, x0_ref)          # the last step ends on the final x0 prediction


@pytest.mark.gpu
@pytest.mark.parametrize("order", [2, 3])
def test_scheduler_step_is_stateful_and_bit_exact(order):
    """step(model_output, t, sample) -> prev_sample, the diffusers contract: the scheduler carries the corrected sample
    and the previous x0 predictions."""
    N, shape = 8, (2, 4, 5, 9)
    s = UniPCMultistepScheduler(**KW, solver_order=order, disable_corrector=[3])
    s.set_timesteps(N, device=DEV)
    o = UO.UniPCOracle(**KW, solver_order=order, disable_corrector=[3])
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
    from oracle import unet_oracle as UNO
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.models import GeneralVAESeg, UNet, unet_init
    o_unet = UNO.build_unet(seed=0)
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
@pytest.mark.parametrize("order", [2, 3])
def test_sampler_vs_oracle(models, order):
    from oracle import ldmseg_oracle as LO
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.trainers import TrainerDiffusion
    B, h, w, T = 2, 16, 24, 5
    rgb = _rgb(B, h, w)
    tr = TrainerDiffusion(p={}, vae_semseg=models["vae"], unet_model=models["unet"],
                          noise_scheduler=UniPCMultistepScheduler(**KW, solver_order=order), args={"gpu": 0})
    lat = tr.sample([""] * B, num_inference_steps=T, seed=42, rgb_latents=rgb)
    ref = LO.sample(models["o_unet"], UO.UniPCOracle(**KW, solver_order=order), rgb, num_inference_steps=T, seed=42)
    assert lat.shape == ref.shape == (B, 4, h, w)
    assert _rel(lat, ref) < 8e-2, _rel(lat, ref)
    # the solver order matters more than the error
    ref1 = LO.sample(models["o_unet"], UO.UniPCOracle(**KW, solver_order=1), rgb, num_inference_steps=T, seed=42)
    assert _rel(ref1, ref) > _rel(lat, ref)
    # return_all_latents: one state per step, the last is the result
    allv = tr.sample([""] * B, num_inference_steps=T, seed=42, rgb_latents=rgb, return_all_latents=True)
    assert allv.shape == (T * B, 4, h, w) and torch.equal(allv[-B:], lat)
    # repeat_noise: every frame starts from the first frame's noise, which comes back with the latents
    rep, noise = tr.sample([""] * B, num_inference_steps=T, seed=42, rgb_latents=rgb, repeat_noise=True)
    first = torch.randn((B, 4, h, w), generator=torch.Generator().manual_seed(42))[0:1].repeat(B, 1, 1, 1)
    assert torch.equal(noise.cpu(), first)
    assert torch.equal(rep, tr.sample([""] * B, num_inference_steps=T, rgb_latents=rgb, noise=first))


@pytest.mark.gpu
def test_graph_replay_equals_eager_and_runs_are_bit_identical(models):
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.trainers import TrainerDiffusion
    B, h, w, T = 2, 16, 24, 6
    rgb = _rgb(B, h, w)
    sched = UniPCMultistepScheduler(**KW, solver_order=3, disable_corrector=[1])
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
    from oracle import unet_oracle as UNO
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

    o_unet = UNO.build_unet(seed=8, cross_attention_dim=768)
    unet = UNet(device=DEV)
    unet.load_state_dict(o_unet.state_dict())
    o_unet = o_unet.to(DEV)
    tok, enc = Tok(), Enc().to(DEV).eval()
    B, h, w, T, g = 2, 16, 24, 4, 4.0
    prompts = ["a car on the road", "two pedestrians"]
    rgb = _rgb(B, h, w)
    sched = UniPCMultistepScheduler(**KW)
    sched.set_timesteps(T)
    tr = TrainerDiffusion(p={}, unet_model=unet, tokenizer=tok, text_encoder=enc, args={"gpu": 0})
    lat = tr.sample(prompts, num_inference_steps=T, guidance_scale=g, seed=42, rgb_latents=rgb, scheduler=sched)
    with torch.no_grad():
        ctx = enc(tok(prompts).input_ids.to(DEV))[0]
        unc = enc(tok([""] * B).input_ids.to(DEV))[0]
    ref = LO.sample(o_unet, UO.UniPCOracle(**KW), rgb, num_inference_steps=T, seed=42, context=ctx,
                    uncond_context=unc, guidance_scale=g)
    ref1 = LO.sample(o_unet, UO.UniPCOracle(**KW), rgb, num_inference_steps=T, seed=42, context=ctx,
                     uncond_context=unc, guidance_scale=1.0)
    assert lat.shape == ref.shape == (B, 4, h, w)
    assert _rel(lat, ref) < 8e-2, _rel(lat, ref)
    assert _rel(ref1, ref) > 2 * _rel(lat, ref)  # the guidance scale matters more than the error


@pytest.mark.gpu
def test_sampler_rejects_self_condition(models):
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.trainers import TrainerDiffusion
    rgb = _rgb(1, 16, 24)
    tr = TrainerDiffusion(p={"train_kwargs": {"self_condition": True}}, unet_model=models["unet"],
                          noise_scheduler=UniPCMultistepScheduler(**KW), args={"gpu": 0})
    with pytest.raises(NotImplementedError, match="self_condition"):
        tr.sample([""], num_inference_steps=4, seed=0, rgb_latents=rgb)


@pytest.mark.gpu
def test_compute_pq_with_unipc_scheduler(models):
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
                          noise_scheduler=UniPCMultistepScheduler(**KW), args={"gpu": 0})
    res = tr.compute_metrics(["pq"], seed=42, dataloader=batches, num_inference_steps=T)
    assert tr.noise_scheduler.timesteps.numel() == T
    ev = EO.CityscapesPQOracle()
    for data, cleaned in zip(batches, tr.last_cleaned):
        for b in range(B):
            ev.add_image(cleaned[b].cpu().numpy().astype(np.int64), data["semseg"][b].numpy())
    want = ev.evaluate()
    for k in ("pq", "sq", "rq", "tp", "fp", "fn", "iou_sum"):
        assert res[k] == want[k], k
