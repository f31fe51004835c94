"""GPU parity of the host mirrors (UNet, seg-AE decoder, scheduler, sampler, integer tail, evaluators) against the
oracle restatements and the golden fixtures generated from the real reference. Everything under test goes through
the C ABI; the oracle is only the checker (it runs its plain PyTorch fp32 modules on the same device for speed).

Stated tolerances (bf16 storage, fp32 accumulate vs fp32 oracle):
  UNet epsilon, one step  : relative L2 <= 3e-2, max-abs <= 0.15 * max|ref|
  seg-AE logits           : relative L2 <= 3e-2
  DDIM update             : bit-exact (fp32)
  sampler, T DDIM steps   : relative L2 <= 8e-2 on the final latents
  panoptic ids / PQ / DVPQ: bit-exact given identical logits / ids
"""
import json
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GOLD = json.load(open(os.path.join(G, "golden.json")))
SCHED_KW = dict(num_train_timesteps=1000, beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear",
                clip_sample=False, set_alpha_to_one=False, steps_offset=1, prediction_type="epsilon", weight="none")
DEV = "cuda"


def _rel(got, ref):
    got, ref = got.float(), ref.float()
    return ((got - ref).pow(2).sum().sqrt() / (ref.pow(2).sum().sqrt() + 1e-12)).item()


@pytest.fixture(scope="module")
def models():
    from oracle import ldmseg_oracle as LO
    from oracle import unet_oracle as UO
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.models import GeneralVAESeg, UNet
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.models import unet_init
    o_unet = UO.build_unet(seed=0)  # full SD-1.4 width, random init, 8-channel conv_in
    unet = UNet(device=DEV)
    unet.load_state_dict(o_unet.state_dict())
    unet.remove_cross_attention()
    o_unet = o_unet.to(DEV)
    kw = dict(in_channels=16, int_channels=256, out_channels=128, latent_channels=4, num_upscalers=2,
              upscale_channels=256, norm_num_groups=32, scaling_factor=0.2)
    o_vae = LO.SegDecoderOracle(**kw)
    sd = unet_init.random_seg_decoder_state_dict(seed=1, **kw)
    g = torch.Generator().manual_seed(9)
    for k in sd:  # non-trivial norm affine parameters
        if sd[k].dim() == 1:
            sd[k] = sd[k] + 0.1 * torch.randn(sd[k].shape, generator=g)
    o_vae.load_state_dict(sd)
    vae = GeneralVAESeg(**kw, device=DEV)
    vae.load_state_dict(sd)
    return dict(o_unet=o_unet, unet=unet, o_vae=o_vae.to(DEV).eval(), vae=vae)


def test_scheduler_step_bit_exact_with_reference_fixture():
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.schedulers import DDIMNoiseScheduler
    z = np.load(os.path.join(G, "ddim_steps.npz"))
    s = DDIMNoiseScheduler(**SCHED_KW)
    s.set_timesteps_inference(50)
    s.move_timesteps_to(DEV)
    eps, x = torch.from_numpy(z["eps"]).to(DEV), torch.from_numpy(z["x"]).to(DEV)
    for t in (999, 499, 19):
        idx = s.timesteps.tolist().index(t)
        for ts in (s.timesteps[idx], t, torch.tensor(t)):  # CUDA 0-dim tensor (the sampler's case), int, CPU tensor
            o = s.step(eps, ts, x)
            assert np.array_equal(o.prev_sample.cpu().numpy(), z[f"prev_{t}"])
            assert np.array_equal(o["pred_original_sample"].cpu().numpy(), z[f"x0_{t}"])


def test_scheduler_step_clip_sample_bit_exact_with_reference_fixture():
    """ldm_ddim_step_clip: clip_sample=True (the reference constructor's default) with two ranges, with and without
    use_clipped_model_output, against vectors of the real reference scheduler (make_golden_ddim_clip.py)."""
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.schedulers import DDIMNoiseScheduler
    z = np.load(os.path.join(G, "ddim_steps_clip.npz"))
    eps, x = torch.from_numpy(z["eps"]).to(DEV), torch.from_numpy(z["x"]).to(DEV)
    for rng in (1.0, 0.5):
        s = DDIMNoiseScheduler(**dict(SCHED_KW, clip_sample=True, clip_sample_range=rng))
        s.set_timesteps_inference(50)
        for t in (999, 499, 19):
            for ucm in (False, True):
                o = s.step(eps, t, x, use_clipped_model_output=ucm)
                tag = f"r{rng}_t{t}_u{int(ucm)}"
                assert np.array_equal(o.prev_sample.cpu().numpy(), z["prev_" + tag]), tag
                assert np.array_equal(o.pred_original_sample.cpu().numpy(), z["x0_" + tag]), tag
    with pytest.raises(Exception):
        DDIMNoiseScheduler(**dict(SCHED_KW, clip_sample=True, clip_sample_range=0.0)).step(eps, 999, x)


def test_seg_decoder_small_reference_fixture():
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.models import GeneralVAESeg
    z = np.load(os.path.join(G, "seg_decoder_small.npz"))
    cfg = GOLD["seg_decoder_small"]["cfg"]
    vae = GeneralVAESeg(**cfg, device=DEV)
    vae.load_state_dict({k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd.")})
    zz = torch.from_numpy(z["z"]).to(DEV)
    lo = vae.decode(zz, interpolate=False)
    hi = vae.decode(zz, interpolate=True)
    assert lo.shape == z["logits_lo"].shape and hi.shape == z["logits_hi"].shape
    assert _rel(lo.cpu(), torch.from_numpy(z["logits_lo"])) < 3e-2
    assert _rel(hi.cpu(), torch.from_numpy(z["logits_hi"])) < 3e-2


def test_seg_encoder_reference_fixture():
    """encode / posterior / forward of the seg-AE against the real reference (tests/golden/seg_encoder_small.npz)."""
    import ast
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.models import GeneralVAESeg
    z = {k: f[k] for name in ("seg_encoder_small.npz", "seg_encoder_small_part2.npz")
         for f in [np.load(os.path.join(G, name))] for k in f.files}
    cfg = ast.literal_eval(str(z["cfg"]))
    vae = GeneralVAESeg(**cfg, device=DEV)
    vae.load_state_dict({k[3:]: torch.from_numpy(v) for k, v in z.items() if k.startswith("sd.")})
    bits = torch.from_numpy(z["bits"]).to(DEV)
    post = vae.encode(bits).latent_dist
    assert post.parameters.shape == z["moments"].shape
    assert _rel(post.parameters.cpu(), torch.from_numpy(z["moments"])) < 3e-2
    assert _rel(post.mode().cpu(), torch.from_numpy(z["mode"])) < 3e-2
    assert _rel(post.std.cpu(), torch.from_numpy(z["std"])) < 3e-2
    out = vae(bits, sample_posterior=False)
    assert list(out.keys()) == ["sample", "posterior"] and out.sample.shape == z["forward"].shape
    assert _rel(out.sample.cpu(), torch.from_numpy(z["forward"])) < 4e-2
    smp = post.sample(generator=torch.Generator(device=DEV).manual_seed(0))
    assert smp.shape == post.mode().shape and torch.isfinite(smp).all()
    with pytest.raises(Exception):
        vae.encode(bits.cpu())  # no CPU fallback


def test_seg_encoder_frame_size_vs_oracle():
    """The default seg-AE (base.yaml:14-33) on the bit planes of one 384x1248 frame against the fp32 oracle."""
    from oracle import ldmseg_oracle as LO
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.models import GeneralVAESeg
    kw = dict(in_channels=16, int_channels=256, out_channels=128, latent_channels=4, num_upscalers=2,
              upscale_channels=256, norm_num_groups=32, scaling_factor=0.2)
    torch.manual_seed(21)
    o_enc = LO.SegEncoderOracle(**kw).eval()
    sd = {k: v.clone() for k, v in o_enc.state_dict().items()}
    sd.update({k: v for k, v in LO.SegDecoderOracle(**kw).state_dict().items()})
    vae = GeneralVAESeg(**kw, device=DEV)
    vae.load_state_dict(sd)
    g = torch.Generator().manual_seed(22)
    bits = ((torch.rand((1, 16, 384, 1248), generator=g) < 0.5).float() * 2 - 1).to(DEV)
    got = vae.encode(bits).latent_dist.parameters
    with torch.no_grad():
        ref = o_enc.to(DEV).encode(bits)
    assert got.shape == ref.shape == (1, 8, 48, 156)
    assert _rel(got, ref) < 3e-2


def test_seg_decoder_full_size_vs_oracle(models):
    zz = torch.randn((2, 4, 12, 39), generator=torch.Generator().manual_seed(3)).to(DEV)
    got = models["vae"].decode(zz)
    with torch.no_grad():
        ref = models["o_vae"].decode(zz)
    assert got.shape == ref.shape == (2, 128, 96, 312)
    assert _rel(got, ref) < 3e-2


@pytest.mark.parametrize("shape", [(2, 16, 24), (1, 12, 39)])
def test_unet_eps_vs_oracle(models, shape):
    B, h, w = shape
    g = torch.Generator().manual_seed(11)
    x = torch.randn((B, 8, h, w), generator=g).to(DEV)
    for t in (999, 499, 19):
        ts = torch.tensor(t, device=DEV)
        out = models["unet"](x, ts, encoder_hidden_states=None)
        assert list(out.keys()) == ["sample"] and out.sample.shape == (B, 4, h, w) and out.sample.dtype == torch.float32
        with torch.no_grad():
            ref = models["o_unet"](x, ts, encoder_hidden_states=None)
        rel = _rel(out.sample, ref)
        mx = (out.sample - ref).abs().max().item() / ref.abs().max().item()
        assert rel < 3e-2 and mx < 0.15, (shape, t, rel, mx)
    tup = models["unet"](x, ts, None, return_dict=False)
    assert isinstance(tup, tuple) and torch.equal(tup[0], out.sample)  # graph replay is deterministic


@pytest.mark.parametrize("shape,t", [((1, 48, 156), 499), ((1, 96, 312), 999)])
def test_unet_eps_frame_sizes_vs_oracle(models, shape, t):
    """One frame at the latent sizes of BASELINE.json: 384x1248 (configs[0..3]: 7 488 tokens at the first level) and
    768x2496 (configs[4]: 29 952 tokens, attention-dominated). The oracle materialises the score matrices in fp32
    (29 GB at the larger size), so one image and one timestep each."""
    B, h, w = shape
    x = torch.randn((B, 8, h, w), generator=torch.Generator().manual_seed(12)).to(DEV)
    ts = torch.tensor(t, device=DEV)
    out = models["unet"](x, ts, encoder_hidden_states=None)
    with torch.no_grad():
        ref = models["o_unet"](x, ts, encoder_hidden_states=None)
    rel = _rel(out.sample, ref)
    mx = (out.sample - ref).abs().max().item() / ref.abs().max().item()
    del ref
    torch.cuda.empty_cache()
    assert out.sample.shape == (B, 4, h, w) and rel < 3e-2 and mx < 0.15, (shape, t, rel, mx)


def test_unet_layernorm_fold_option_vs_oracle(models):
    """UNet.ln_fold = True (LayerNorm folded into the QKV / GEGLU GEMMs, off by default because it measured slower):
    same tolerance against the oracle as the default path, and no further from it than the default path is."""
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.models import UNet
    unet = UNet(device=DEV)
    unet.ln_fold = True
    unet.load_state_dict(models["o_unet"].state_dict())
    unet.remove_cross_attention()
    B, h, w = 2, 16, 24
    x = torch.randn((B, 8, h, w), generator=torch.Generator().manual_seed(13)).to(DEV)
    ts = torch.tensor(499, device=DEV)
    got = unet(x, ts, encoder_hidden_states=None).sample
    base = models["unet"](x, ts, encoder_hidden_states=None).sample
    with torch.no_grad():
        ref = models["o_unet"](x, ts, encoder_hidden_states=None)
    rel, rel_base = _rel(got, ref), _rel(base, ref)
    assert rel < 3e-2 and rel <= 1.5 * rel_base + 1e-3, (rel, rel_base)
    assert not torch.equal(got, base)  # the option really took the other path


def test_sampler_vs_oracle(models):
    from oracle import ldmseg_oracle as LO
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.schedulers import DDIMNoiseScheduler
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.trainers import TrainerDiffusion
    B, h, w, T = 2, 16, 24, 4
    rgb = (0.18215 * torch.randn((B, 4, h, w), generator=torch.Generator().manual_seed(1234))).to(DEV)
    sched = DDIMNoiseScheduler(**SCHED_KW)
    tr = TrainerDiffusion(p={}, vae_semseg=models["vae"], unet_model=models["unet"], noise_scheduler=sched,
                          args={"gpu": 0})
    lat = tr.sample([""] * B, num_inference_steps=T, seed=42, rgb_latents=rgb)
    ref = LO.sample(models["o_unet"], LO.DDIMOracle(), rgb, num_inference_steps=T, seed=42)
    assert lat.shape == ref.shape == (B, 4, h, w)
    assert _rel(lat, ref) < 8e-2
    lat2 = tr.sample([""] * B, num_inference_steps=T, seed=42, rgb_latents=rgb)
    assert torch.equal(lat, lat2)  # same seed -> identical latents (CPU generator noise, deterministic kernels)
    # decode_latents keeps the reference contract: NCHW fp32 logits at the input resolution
    logits = tr.decode_latents(lat, return_logits=True)
    assert logits.shape == (B, 128, 8 * h, 8 * w) and logits.dtype == torch.float32
    ref_logits = LO.decode_latents(models["o_vae"], lat)
    assert _rel(logits, ref_logits) < 3e-2


def test_sampler_self_condition_vs_oracle():
    """H1 with train_kwargs.self_condition=True (trainers_ldm_cond.py:1135-1136,1152-1153): the 12-channel conv_in reads
    x_t, rgb_latents and the previous step's pred_original_sample; cond weights random so the branch matters."""
    from oracle import ldmseg_oracle as LO
    from oracle import unet_oracle as UO
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.models import UNet
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.schedulers import DDIMNoiseScheduler
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.trainers import TrainerDiffusion
    mk = dict(in_channels=8, init_mode_seg="copy", init_mode_image="copy", cond_channels=4, init_mode_cond="random")
    o_unet = UO.build_unet(seed=3, model_kwargs=mk)
    assert o_unet.conv_in.weight.shape[1] == 12
    unet = UNet(device=DEV)
    unet.load_state_dict(o_unet.state_dict())
    unet.remove_cross_attention()
    o_unet = o_unet.to(DEV)
    B, h, w, T = 2, 16, 24, 4
    rgb = (0.18215 * torch.randn((B, 4, h, w), generator=torch.Generator().manual_seed(1234))).to(DEV)
    tr = TrainerDiffusion(p={"train_kwargs": {"self_condition": True}}, unet_model=unet,
                          noise_scheduler=DDIMNoiseScheduler(**SCHED_KW), args={"gpu": 0})
    lat = tr.sample([""] * B, num_inference_steps=T, seed=42, rgb_latents=rgb)
    ref = LO.sample(o_unet, LO.DDIMOracle(), rgb, num_inference_steps=T, seed=42, self_condition=True)
    assert _rel(lat, ref) < 8e-2


@pytest.fixture(scope="module")
def vae_image():
    from oracle import vae_image_oracle as VO
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.models import GeneralVAEImage
    o = VO.build_vae_image(seed=5)
    g = torch.Generator().manual_seed(11)
    sd = o.state_dict()
    for k in sd:  # non-trivial norm affine parameters and biases
        if sd[k].dim() == 1:
            sd[k] = sd[k] + 0.1 * torch.randn(sd[k].shape, generator=g)
    o.load_state_dict(sd)
    assert sum(p.numel() for p in o.parameters()) == 34163664  # SD-1.4 VAE encoder + quant_conv
    m = GeneralVAEImage.from_pretrained(state_dict=sd, device=DEV)
    m.set_scaling_factor(0.18215)
    return dict(o=o.to(DEV), m=m)


@pytest.mark.parametrize("shape", [(2, 64, 128), (1, 384, 1248)])
def test_vae_image_encoder_vs_oracle(vae_image, shape):
    """SURVEY 8f rank 1: moments of the RGB VAE encoder (+ quant_conv) against the restated diffusers AutoencoderKL,
    at a small size and at the 384x1248 frame size (7 488-token single-head attention in the mid block)."""
    B, H, W = shape
    x = torch.rand((B, 3, H, W), generator=torch.Generator().manual_seed(21)).to(DEV)
    xin = 2. * x - 1.
    with torch.no_grad():
        ref = vae_image["o"].moments(xin)
    got = vae_image["m"].encode_moments(xin)
    assert got.shape == ref.shape == (B, 8, H // 8, W // 8) and got.dtype == torch.float32
    assert _rel(got, ref) < 3e-2, _rel(got, ref)
    dist = vae_image["m"].encode(xin).latent_dist
    assert torch.equal(dist.mode(), got[:, :4])
    assert dist.sample().shape == (B, 4, H // 8, W // 8)
    # the fused affine map of encode_inputs gives the same moments as the explicit 2x - 1
    got2 = vae_image["m"].encode_moments(x, scale=2.0, shift=-1.0)
    assert torch.equal(got2, got)


def test_encode_inputs_vs_oracle(vae_image):
    """trainers_ldm_cond.py:336-396: resize of the image, 2x - 1, mode of the posterior, resize of the latents, scaling."""
    from oracle import vae_image_oracle as VO
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.trainers import TrainerDiffusion
    x = torch.rand((2, 3, 96, 200), generator=torch.Generator().manual_seed(22)).to(DEV)
    tr = TrainerDiffusion(p={"latent_size": (6, 20)}, vae_image=vae_image["m"], args={"gpu": 0})
    lat, mean = tr.encode_inputs(x, resize=(64, 128))
    ref, ref_mean = VO.encode_inputs(vae_image["o"], x, resize=(64, 128), latent_size=(6, 20))
    assert lat.shape == ref.shape == (2, 4, 6, 20)
    assert _rel(lat, ref) < 3e-2 and torch.equal(lat, mean)
    lat2, _ = tr.encode_inputs(x[:, :, :64, :128].contiguous(), resize=None)  # no resize at all
    ref2, _ = VO.encode_inputs(vae_image["o"], x[:, :, :64, :128])
    assert lat2.shape == (2, 4, 8, 16) and _rel(lat2, ref2) < 3e-2


def test_unet_cross_attention_vs_oracle():
    """SURVEY 8f rank 4: the UNet with its cross-attention layers kept (SD-1.4 cross_attention_dim 768). (a) explicit
    encoder_hidden_states of 77 tokens (the CLIP text context length); (b) the 'learnable' descriptor variant
    (descriptors.py:89-91, unet.py:322-323): 128 object queries are the context and the sampler needs no extra input."""
    from oracle import ldmseg_oracle as LO
    from oracle import unet_oracle as UO
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.models import UNet
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.schedulers import DDIMNoiseScheduler
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.trainers import TrainerDiffusion
    g = torch.Generator().manual_seed(5)
    B, h, w = 2, 16, 24
    x = torch.randn((B, 8, h, w), generator=g).to(DEV)
    t = torch.tensor(499, device=DEV)
    # (a) explicit context
    o_unet = UO.build_unet(seed=4, cross_attention_dim=768)
    unet = UNet(device=DEV)
    unet.load_state_dict(o_unet.state_dict())
    o_unet = o_unet.to(DEV)
    ehs = torch.randn((B, 77, 768), generator=g).to(DEV)
    with torch.no_grad():
        ref = o_unet(x, t, encoder_hidden_states=ehs)
        ref0 = o_unet(x, t, encoder_hidden_states=torch.zeros_like(ehs))
    got = unet(x, t, encoder_hidden_states=ehs).sample
    assert _rel(got, ref) < 3e-2, _rel(got, ref)
    assert _rel(ref0, ref) > 3 * _rel(got, ref)  # the context moves the output by more than the error
    got_b = unet(x, t, encoder_hidden_states=0.5 * ehs).sample  # a new context re-projects k / v of every layer
    with torch.no_grad():
        ref_b = o_unet(x, t, encoder_hidden_states=0.5 * ehs)
    assert _rel(got_b, ref_b) < 3e-2
    with pytest.raises(ValueError):
        unet(x, t, encoder_hidden_states=None)
    del unet, o_unet
    # (b) learnable object queries, through the sampler
    o_unet = UO.build_unet(seed=6, cross_attention_dim=768, learnable_queries=(128, 768))
    unet = UNet(device=DEV)
    unet.load_state_dict(o_unet.state_dict())
    o_unet = o_unet.to(DEV)
    rgb = (0.18215 * torch.randn((B, 4, h, w), generator=torch.Generator().manual_seed(1234))).to(DEV)
    tr = TrainerDiffusion(p={}, unet_model=unet, noise_scheduler=DDIMNoiseScheduler(**SCHED_KW), args={"gpu": 0})
    lat = tr.sample([""] * B, num_inference_steps=3, seed=42, rgb_latents=rgb)
    ref = LO.sample(o_unet, LO.DDIMOracle(), rgb, num_inference_steps=3, seed=42)
    assert _rel(lat, ref) < 8e-2, _rel(lat, ref)


class _ToyTokenizer:
    """Stands in for CLIPTokenizer (a third-party model the reference loads, descriptors.py:99-101): same call contract."""
    model_max_length = 12

    def __call__(self, texts, padding="max_length", max_length=None, truncation=True, return_tensors="pt"):
        from types import SimpleNamespace
        L_ = max_length or self.model_max_length
        ids = torch.zeros((len(texts), L_), dtype=torch.long)
        for i, t in enumerate(texts):
            codes = [1 + (ord(c) % 60) for c in t][:L_]
            ids[i, :len(codes)] = torch.tensor(codes, dtype=torch.long)
        return SimpleNamespace(input_ids=ids)


class _ToyTextEncoder(torch.nn.Module):
    """Stands in for CLIPTextModel: input_ids -> (last_hidden_state [B, L, 768],)."""

    def __init__(self):
        super().__init__()
        torch.manual_seed(12)
        self.emb = torch.nn.Embedding(64, 768)
        self.pos = torch.nn.Parameter(0.1 * torch.randn(12, 768))

    def forward(self, input_ids):
        return (self.emb(input_ids) + self.pos[None, :input_ids.shape[1]],)


def _clip_text_model():
    """The class the reference loads (descriptors.py:100: transformers.CLIPTextModel), SD-1.4's text-encoder geometry
    (768 wide, 77 positions, 49 408 tokens) with two layers, random-init (no checkpoint offline)."""
    from transformers import CLIPTextConfig, CLIPTextModel
    torch.manual_seed(13)
    cfg = CLIPTextConfig(hidden_size=768, intermediate_size=3072, num_attention_heads=12, num_hidden_layers=2,
                         max_position_embeddings=77, vocab_size=49408)
    return CLIPTextModel(cfg)


class _ClipLengthTokenizer(_ToyTokenizer):
    model_max_length = 77


@pytest.mark.parametrize("encoder", ["toy", "transformers_clip"])
def test_sampler_classifier_free_guidance_vs_oracle(encoder):
    """H1 with a text encoder (trainers_ldm_cond.py:1110-1122,1126-1129,1147-1149): doubled batch [uncond | text],
    encoder_hidden_states through the kept cross-attention, guidance fused into the DDIM kernel. Once with a toy
    encoder, once with transformers' CLIPTextModel (the reference's class) and its 77-token context."""
    from oracle import ldmseg_oracle as LO
    from oracle import unet_oracle as UO
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.models import UNet
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.schedulers import DDIMNoiseScheduler
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.trainers import TrainerDiffusion
    o_unet = UO.build_unet(seed=8, cross_attention_dim=768)
    unet = UNet(device=DEV)
    unet.load_state_dict(o_unet.state_dict())
    o_unet = o_unet.to(DEV)
    if encoder == "toy":
        tok, enc = _ToyTokenizer(), _ToyTextEncoder().to(DEV).eval()
    else:
        tok, enc = _ClipLengthTokenizer(), _clip_text_model().to(DEV).eval()
    B, h, w, T, g = 2, 16, 24, 3, 4.0
    prompts = ["a car on the road", "two pedestrians"]
    rgb = (0.18215 * torch.randn((B, 4, h, w), generator=torch.Generator().manual_seed(1234))).to(DEV)
    tr = TrainerDiffusion(p={}, unet_model=unet, tokenizer=tok, text_encoder=enc,
                          noise_scheduler=DDIMNoiseScheduler(**SCHED_KW), args={"gpu": 0})
    lat = tr.sample(prompts, num_inference_steps=T, guidance_scale=g, seed=42, rgb_latents=rgb)
    with torch.no_grad():
        ctx = enc(tok(prompts).input_ids.to(DEV))[0]
        unc = enc(tok([""] * B).input_ids.to(DEV))[0]
    ref = LO.sample(o_unet, LO.DDIMOracle(), rgb, num_inference_steps=T, seed=42, context=ctx, uncond_context=unc,
                    guidance_scale=g)
    ref1 = LO.sample(o_unet, LO.DDIMOracle(), rgb, num_inference_steps=T, seed=42, context=ctx, uncond_context=unc,
                     guidance_scale=1.0)
    assert lat.shape == ref.shape == (B, 4, h, w)
    assert _rel(lat, ref) < 8e-2, _rel(lat, ref)
    assert _rel(ref1, ref) > 2 * _rel(lat, ref)  # the guidance scale matters more than the error
    # a UNet whose cross-attention was removed ignores the descriptors, as the reference's does (attn2 is None)
    unet.remove_cross_attention()
    lat0 = tr.sample(prompts, num_inference_steps=T, guidance_scale=g, seed=42, rgb_latents=rgb)
    assert lat0.shape == (B, 4, h, w) and torch.isfinite(lat0).all() and not torch.equal(lat0, lat)


def test_sampler_clip_image_descriptors_vs_oracle():
    """image_descriptors == 'clip_image' (descriptors.py:15-31,67-71; trainers_ldm_cond.py:1102-1109,665-677):
    transformers' CLIPVisionModel (ViT-L/14 geometry, two layers, random init) -> 257 x 1024 descriptors ->
    encoder_hid_proj 1024 -> 768 -> cross-attention. The reference doubles the batch with the SAME descriptors in both
    halves; the mirror computes one half (uncond + g * (text - uncond) == uncond)."""
    from transformers import CLIPVisionConfig, CLIPVisionModel
    from oracle import ldmseg_oracle as LO
    from oracle import unet_oracle as UO
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.models import UNet
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.schedulers import DDIMNoiseScheduler
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.trainers import TrainerDiffusion

    class MyCLIPVisionModel(torch.nn.Module):  # the reference's wrapper (descriptors.py:15-31), by composition
        def __init__(self, cfg):
            super().__init__()
            self.clip = CLIPVisionModel(cfg)

        def forward(self, pixel_values=None, **kw):
            out = self.clip.vision_model(pixel_values=pixel_values)
            return {"last_feat": out.last_hidden_state.permute(0, 2, 1)}

    torch.manual_seed(14)
    vis = MyCLIPVisionModel(CLIPVisionConfig(hidden_size=1024, intermediate_size=4096, num_attention_heads=16,
                                             num_hidden_layers=2, image_size=224, patch_size=14)).to(DEV).eval()
    o_unet = UO.build_unet(seed=9, cross_attention_dim=768)
    torch.manual_seed(15)
    o_unet.modify_encoder_hidden_state_proj(1024, 768)          # descriptors.py:71
    unet = UNet(device=DEV)
    unet.load_state_dict(o_unet.state_dict())
    o_unet = o_unet.to(DEV)
    B, h, w, T = 2, 16, 24, 2
    images = torch.rand((B, 3, 8 * h, 8 * w), generator=torch.Generator().manual_seed(3)).to(DEV)
    rgb = (0.18215 * torch.randn((B, 4, h, w), generator=torch.Generator().manual_seed(1234))).to(DEV)
    tr = TrainerDiffusion(p={}, unet_model=unet, image_descriptor_model=vis,
                          noise_scheduler=DDIMNoiseScheduler(**SCHED_KW), args={"gpu": 0})
    lat = tr.sample([""] * B, num_inference_steps=T, guidance_scale=7.5, seed=42, rgb_latents=rgb, rgb_images=images)
    with torch.no_grad():
        x = F.interpolate(images, size=(224, 224), mode="bilinear", align_corners=False)
        mean = torch.tensor([0.48145466, 0.4578275, 0.40821073], device=DEV).view(1, 3, 1, 1)
        std = torch.tensor([0.26862954, 0.26130258, 0.27577711], device=DEV).view(1, 3, 1, 1)
        d = vis((x - mean) / std)["last_feat"]
        desc = d.view(d.shape[0], d.shape[1], -1).permute(0, 2, 1).float()
    assert desc.shape == (B, 257, 1024)
    ref = LO.sample(o_unet, LO.DDIMOracle(), rgb, num_inference_steps=T, seed=42, context=desc, uncond_context=desc,
                    guidance_scale=7.5)   # the reference's doubled batch with identical halves
    assert _rel(lat, ref) < 8e-2, _rel(lat, ref)


def test_tail_ids_bit_exact_given_identical_logits(models):
    """H6/H7: feed the SAME fp32 logits to the CUDA tail and to the restated reference tail."""
    from oracle import ldmseg_oracle as LO
    from video_latent_diffusion_panoptic_segmentation_b200 import ops
    B, h, w, C = 2, 48, 156, 128
    g = torch.Generator().manual_seed(77)
    lo = torch.randn((B, h, w, C), generator=g) * 1.5
    # a few confident blobs so that segments survive count_th / overlap_th, plus low-confidence background; the blob
    # channels are pushed negative elsewhere so that their sigmoid area (the overlap denominator) is the blob itself
    lo[..., 10:14] -= 5.0
    for k, (y0, x0, hh, ww) in enumerate([(2, 3, 20, 40), (25, 60, 20, 50), (5, 100, 30, 50), (30, 5, 15, 40)]):
        lo[:, y0:y0 + hh, x0:x0 + ww, 10 + k] += 14.0
    # one more blob whose channel is positive over most of the image -> argmax area / sigmoid area < overlap_th
    lo[..., 20] += 1.0
    lo[:, 36:46, 100:150, 20] += 9.0
    lo = lo.to(DEV)
    ids = torch.empty((B, 2 * h, 2 * w), dtype=torch.int32, device=DEV)
    counts = torch.empty((B, 2, C), dtype=torch.int32, device=DEV)
    cleaned = torch.empty_like(ids)
    ops.logits_to_ids(lo, ids, counts, up=2, mask_th=0.5, ignore_label=127)
    ops.segment_filter(ids, counts, cleaned, count_th=512, overlap_th=0.5, ignore_label=127)
    full = F.interpolate(lo.permute(0, 3, 1, 2).cpu(), scale_factor=2, mode="bilinear", align_corners=False)
    kept_total = 0
    for b in range(B):
        pred, cl, kept = LO.logits_to_panoptic(full[b], 0.5, 512, 0.5, 127)
        assert np.array_equal(pred, ids[b].cpu().numpy())
        assert np.array_equal(cl, cleaned[b].cpu().numpy())
        kept_total += len(kept)
    assert kept_total >= 4


def test_bit_decode_reference_sample_outputs():
    from video_latent_diffusion_panoptic_segmentation_b200 import ops
    z = np.load(os.path.join(G, "bitmap_sample_outputs.npz"))
    bits = torch.from_numpy(z["bits_u8"].astype(np.float32) / 255.0)[None].to(DEV)  # {0, 0.498, 1.0}
    ids = torch.empty((1,) + z["semseg"].shape, dtype=torch.int32, device=DEV)
    ops.decode_bitmap(bits.contiguous(), ids, quirk31=True)
    assert np.array_equal(ids[0].cpu().numpy(), z["decoded"])
    enc = torch.empty_like(bits)
    ops.encode_bitmap(torch.from_numpy(z["semseg"].astype(np.int32))[None].to(DEV), enc, ignore_label=0, fill=0.5)
    assert np.array_equal((enc[0].cpu().numpy() * 255).astype(np.uint8), z["bits_u8"])


def test_vpq_eval_matches_reference_golden():
    from synth import vpq_case
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.evaluations import aggregate, vpq_eval
    rows = []
    for case in GOLD["vpq"].values():
        pred, gt = vpq_case(case["seed"], case["H"], case["W"])
        out = vpq_eval([pred, gt])
        for a, b in zip(out, case["out"]):
            assert a.tolist() == b
        rows.append(out)
        gt64 = (gt // 2 ** 20) * 64 + (gt % 2 ** 20) % 64
        pr64 = (pred // 2 ** 20) * 64 + (pred % 2 ** 20) % 64
        for a, b in zip(vpq_eval([pr64, gt64], max_ins=64, guard_union=True), case["out64"]):
            assert a.tolist() == b
    from oracle import eval_oracle as EO
    agg, ref = aggregate(rows), EO.dvpq_aggregate(rows)
    assert agg["pq"] == ref["pq"] and agg["pq_things"] == ref["pq_things"] and agg["pq_stuff"] == ref["pq_stuff"]


def test_cityscapes_evaluator_matches_reference_golden():
    from synth import city_case
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.evaluations import CityscapesPanopticEvaluator
    ev = CityscapesPanopticEvaluator(thing_ids={11, 12, 13, 14, 15, 16, 17, 18}, device=DEV)
    for img in GOLD["cityscapes_pq"]["images"]:
        pred, gt = city_case(img["seed"])
        ev.add_image(pred, gt)
        assert (ev.TP, ev.FP, ev.FN) == (img["tp"], img["fp"], img["fn"])
        assert ev.iou_sum == img["iou_sum"]
    res, want = ev.evaluate(), GOLD["cityscapes_pq"]["result"]
    for k in ("pq", "sq", "rq", "tp", "fp", "fn", "iou_sum", "thing_pq", "thing_sq", "thing_rq", "stuff_pq",
              "stuff_sq", "stuff_rq"):
        assert res[k] == want[k], k
    assert {str(c): m for c, m in res["per_class"].items()} == want["per_class"]


@pytest.mark.parametrize("which", ["vpq", "city"])
def test_evaluator_edge_cases_match_reference_golden(which):
    """tests/golden/edge_cases.json holds the REAL reference's outputs on the edge inputs of tests/synth.py (identical
    maps, nothing matches, all-void / all-ignore ground truth, all-void prediction, one pixel, > 1 000 distinct id
    pairs -- the joint-histogram table has to grow --, IoU exactly 0.5, 512 one-pixel components, a split thing)."""
    from synth import edge_cases_city, edge_cases_vpq
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.evaluations import CityscapesPanopticEvaluator, vpq_eval
    edge = json.load(open(os.path.join(G, "edge_cases.json")))
    if which == "vpq":
        for name, (pred, gt) in edge_cases_vpq().items():
            for a, b in zip(vpq_eval([pred, gt]), edge["vpq"][name]):
                assert a.tolist() == b, name
    else:
        for name, (pred, gt) in edge_cases_city().items():
            ev = CityscapesPanopticEvaluator(thing_ids={11, 12, 13, 14, 15, 16, 17, 18}, device=DEV)
            ev.add_image(pred, gt)
            res, want = ev.evaluate(), edge["city"][name]
            assert (ev.TP, ev.FP, ev.FN, ev.iou_sum) == (want["tp"], want["fp"], want["fn"], want["iou_sum"]), name
            assert (res["pq"], res["sq"], res["rq"]) == (want["pq"], want["sq"], want["rq"]), name
            assert {str(c): m for c, m in res["per_class"].items()} == want["per_class"], name


def test_compute_pq_end_to_end(models):
    """compute_metrics(['pq']) on synthetic batches; the PQ is re-derived by the oracle evaluator from the ids the
    CUDA path produced (bit-exact statistics), and the ids from the oracle tail on the oracle decoder's logits agree
    with the CUDA ids on >= 99% of pixels (bf16 decoder vs fp32 decoder)."""
    from oracle import eval_oracle as EO
    from synth import synth_panoptic
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.schedulers import DDIMNoiseScheduler
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.trainers import TrainerDiffusion
    B, h, w, T = 2, 16, 24, 3
    H, W = 8 * h, 8 * w
    rng = np.random.default_rng(7)
    batches = []
    for i in range(2):
        rgb = 0.18215 * torch.randn((B, 4, h, w), generator=torch.Generator().manual_seed(1234 + i))
        gts = []
        for _ in range(B):
            _, cat, _ = synth_panoptic(rng, H, W, n_seeds=40)
            cat = cat.astype(np.int64)
            cat[cat == 255] = 0
            gts.append(cat)
        batches.append({"rgb_latents": rgb, "semseg": torch.from_numpy(np.stack(gts)),
                        "mask": torch.ones((B, H, W), dtype=torch.bool)})
    p = {"eval_kwargs": {"mask_th": 0.0, "count_th": 64, "overlap_th": 0.0}, "ignore_label": 127}
    tr = TrainerDiffusion(p=p, vae_semseg=models["vae"], unet_model=models["unet"],
                          noise_scheduler=DDIMNoiseScheduler(**SCHED_KW), args={"gpu": 0})
    res = tr.compute_metrics(["pq"], seed=42, dataloader=batches, num_inference_steps=T)
    ev = EO.CityscapesPQOracle()
    for data, cleaned in zip(batches, tr.last_cleaned):
        for b in range(B):
            ev.add_image(cleaned[b].cpu().numpy().astype(np.int64), data["semseg"][b].numpy())
    want = ev.evaluate()
    for k in ("pq", "sq", "rq", "tp", "fp", "fn", "iou_sum"):
        assert res[k] == want[k], k
    assert res["tp"] + res["fn"] > 0


def test_resized_cropped_tail_vs_reference_chain(models):
    """H5: when the resizes are not the identity (RGB size != decoder size, padding mask, meta.im_size), the CUDA tail
    (bilinear x2 -> bilinear to RGB size -> crop_padding -> bilinear to im_size -> argmax/threshold/merge) follows the
    reference chain of F.interpolate calls (trainers_ldm_cond.py:1264-1325) run by torch on the SAME decoder logits.
    Float resampling differs in the last bits between implementations, so ids may flip on a vanishing share of pixels."""
    from oracle import ldmseg_oracle as LO
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.schedulers import DDIMNoiseScheduler
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.trainers import TrainerDiffusion
    B, h, w = 2, 8, 16
    p = {"eval_kwargs": {"mask_th": 0.3, "count_th": 64, "overlap_th": 0.2}, "ignore_label": 127}
    tr = TrainerDiffusion(p=p, vae_semseg=models["vae"], unet_model=models["unet"],
                          noise_scheduler=DDIMNoiseScheduler(**SCHED_KW), args={"gpu": 0})
    lat = (0.2 * 3.0 * torch.randn((B, 4, h, w), generator=torch.Generator().manual_seed(5))).to(DEV)
    rgb_size = (72, 136)                       # != decoder size 64 x 128
    masks = torch.zeros((B,) + rgb_size, dtype=torch.bool)
    masks[0, :60, :120] = True                 # padded bottom / right
    masks[1, 4:70, 10:130] = True
    im_sizes = [(90, 180), (66, 120)]
    got = tr.panoptic_ids_resized(lat, rgb_size, masks.to(DEV), im_sizes)
    # reference chain on the CUDA decoder's own logits
    logits = models["vae"].decode_nhwc(lat, scale=1.0 / models["vae"].scaling_factor).permute(0, 3, 1, 2).cpu()
    full = F.interpolate(logits, scale_factor=2, mode="bilinear", align_corners=False)
    full = F.interpolate(full, size=rgb_size, mode="bilinear", align_corners=False)
    for b in range(B):
        co = masks[b].nonzero()
        y0, y1, x0, x1 = co[:, 0].min(), co[:, 0].max(), co[:, 1].min(), co[:, 1].max()
        crop = full[b][:, y0:y1 + 1, x0:x1 + 1]
        img = F.interpolate(crop[None].float(), size=im_sizes[b], mode="bilinear", align_corners=False)[0]
        pred, cl, _ = LO.logits_to_panoptic(img, 0.3, 64, 0.2, 127)
        ids, cleaned, _ = got[b]
        assert tuple(ids.shape[-2:]) == im_sizes[b]
        diff = ids[0].cpu().numpy() != pred
        mism = float(diff.mean())
        assert mism < 2e-3, f"image {b}: {mism:.4%} of the ids differ from the reference chain"
        # The integer part is exact wherever the floats decide: an id may only flip where the reference's own logits are
        # a near-tie -- top-2 logit gap or distance of the max probability to mask_th below 1e-3 (the three chained
        # resamplings agree with torch's to ~1e-6 relative; which of two equal-to-the-last-bit candidates wins is not
        # a property of the algorithm).
        top2 = img.topk(2, dim=0).values
        gap = (top2[0] - top2[1]).numpy()
        pmax = F.softmax(img, dim=0).max(dim=0)[0].numpy()
        near = (gap < 1e-3) | (np.abs(pmax - 0.3) < 1e-3)
        assert not (diff & ~near).any(), f"image {b}: {(diff & ~near).sum()} ids differ away from any tie"
        mism_c = float((cleaned[0].cpu().numpy() != cl).mean())
        assert mism_c < 1e-2, f"image {b}: {mism_c:.4%} of the merged ids differ"


def test_clip_dvpq_device_windows_match_reference_logic():
    """SURVEY 8e / H9 on device-resident id maps: windows of k stacked frames through ldm_pan_combine + ldm_joint_hist
    (+ ldm_depth_mask_pred) against the restated eval_dvpq.py window logic (width-concatenated numpy arrays), bit-exact
    for the four per-class arrays; then the whole-clip aggregate for k = 1, 2, 3."""
    from oracle import eval_oracle as EO
    from test_host_cpu import _clip
    from video_latent_diffusion_panoptic_segmentation_b200.eval import clip_dvpq as CD
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.evaluations.new_eval import aggregate
    n_frames = 6
    maps = _clip(n_frames, H=48, W=64, seed=11)
    dev_maps = [torch.from_numpy(m).to(DEV) for m in maps]
    rng = np.random.default_rng(5)
    dg = rng.integers(0, 4000, size=maps[0].shape).astype(np.uint16)
    dg[rng.random(dg.shape) < 0.2] = 0
    dp = (dg.astype(np.float64) * rng.uniform(0.6, 1.5, size=dg.shape)).astype(np.uint16)
    for k in (1, 2, 3):
        rows = [EO.dvpq_window(*[[m[i + j] for j in range(k)] for m in maps]) for i in range(n_frames - k + 1)]
        want = aggregate(rows)
        got = CD.dvpq_clip_sharded(*dev_maps, n_frames=n_frames, eval_frames=k)
        assert got["n_windows"] == n_frames - k + 1
        for key in ("iou", "tp", "fn", "fp"):
            assert np.array_equal(got[key], want[key]), (k, key)
        assert got["pq"] == want["pq"] and got["pq_things"] == want["pq_things"]
    # depth-aware windows (uint16 samples, wrap-around arithmetic of the reference)
    k, th = 2, 0.25
    rows = [EO.dvpq_window(*[[m[i + j] for j in range(k)] for m in maps],
                           depth_pred=[dp[i + j] for j in range(k)], depth_gt=[dg[i + j] for j in range(k)],
                           depth_thres=th) for i in range(n_frames - k + 1)]
    want = aggregate(rows)
    got = CD.dvpq_clip_sharded(*dev_maps, n_frames=n_frames, eval_frames=k,
                               depth_pred=torch.from_numpy(dp.astype(np.int32)).to(DEV),
                               depth_gt=torch.from_numpy(dg.astype(np.int32)).to(DEV), depth_thres=th, depth_bits=16)
    for key in ("iou", "tp", "fn", "fp"):
        assert np.array_equal(got[key], want[key]), ("depth", key)
    assert abs(got["abs_rel"] - want["abs_rel"]) <= 1e-12 * abs(want["abs_rel"])


@pytest.mark.parametrize("variant", ["latents_remove", "images_learnable"])
def test_main_ldm_entry_point(variant):
    """tools/main_ldm.py mirror, eval_only branch, end to end on synthetic frames: (a) the default path (latents handed
    over, cross-attention removed); (b) RGB frames through the VAE encoder + learnable object queries as the UNet's
    cross-attention context. Checks the plumbing (shapes, counters, determinism), not a PQ value: weights are random."""
    import copy
    from video_latent_diffusion_panoptic_segmentation_b200.tools import main_ldm
    p = copy.deepcopy(main_ldm.BASE)
    ov = ["base.sampling_kwargs.num_inference_steps=2", "base.synthetic.frames=2", "base.synthetic.batch_size=2",
          "base.synthetic.size=[64,128]", "base.eval_kwargs.count_th=16"]
    if variant == "images_learnable":
        ov += ["base.synthetic.from_images=True", "base.train_kwargs.image_descriptors=learnable"]
    p = main_ldm.apply_overrides(p, ov)
    res = main_ldm.main_worker(0, 1, dict(main_ldm.DIST), p)
    assert set(("pq", "sq", "rq", "tp", "fp", "fn")) <= set(res)
    assert res["tp"] + res["fn"] > 0  # the synthetic ground truth has segments
    res2 = main_ldm.main_worker(0, 1, dict(main_ldm.DIST), p)
    assert (res2["tp"], res2["fp"], res2["fn"], res2["iou_sum"]) == (res["tp"], res["fp"], res["fn"], res["iou_sum"])


def test_batched_evaluator_equals_stepwise_and_oracle():
    """ldm_city_pan_maps + ldm_joint_hist_batch (one labelling over all thing classes of all images, one histogram launch,
    one D2H) against the step-by-step form (ldm_ccl_label4 per class ...) and the oracle evaluator: pan maps bit-identical,
    statistics bit-identical. Inputs: the seeded city cases, the edge cases, and a speckled 8-image batch in which every
    thing class has hundreds of components (several per warp / per 1024-pixel block, all slots of the rank kernel)."""
    from oracle import eval_oracle as EO
    from synth import city_case, edge_cases_city
    from video_latent_diffusion_panoptic_segmentation_b200 import ops
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.evaluations import CityscapesPanopticEvaluator
    things = {11, 12, 13, 14, 15, 16, 17, 18}
    cases = [city_case(s, 96, 160) for s in (3, 4, 5, 6)] + list(edge_cases_city().values())
    rng = np.random.default_rng(77)
    speck_pred = rng.integers(-1, 24, size=(8, 120, 200)).astype(np.int64)
    speck_gt = np.where(rng.random((8, 120, 200)) < 0.5, speck_pred, rng.integers(0, 24, size=(8, 120, 200)))
    coarse = np.kron(rng.integers(0, 20, size=(8, 15, 25)), np.ones((8, 8), dtype=np.int64))
    speck_pred[:, :, 96:] = coarse[:, :, 96:]             # half speckle, half 8x8 blocks
    for pred, gt in cases + [(speck_pred, speck_gt)]:
        pred3, gt3 = (pred[None], gt[None]) if pred.ndim == 2 else (pred, gt)
        ev_b = CityscapesPanopticEvaluator(thing_ids=things, device=DEV)
        ev_s = CityscapesPanopticEvaluator(thing_ids=things, device=DEV)
        ev_o = EO.CityscapesPQOracle()
        pt = torch.from_numpy(pred3.astype(np.int32)).to(DEV)
        gtt = torch.from_numpy(gt3.astype(np.int32)).to(DEV)
        slots, n_things = ev_b._thing_slots()
        pp, gp = ops.city_pan_maps(pt, gtt, slots, n_things, 0, 1 << 20)
        for b in range(pred3.shape[0]):
            pp_s, gp_s = ev_s.panoptic_maps(pred3[b], gt3[b])
            assert torch.equal(pp[b], pp_s) and torch.equal(gp[b], gp_s)
            ev_s.add_image_stepwise(pred3[b], gt3[b])
            if b < 2:   # (the oracle paints one boolean mask per component: two images of the speckled batch suffice)
                pp_o, gp_o = ev_o.panoptic_maps(pred3[b].copy(), gt3[b])
                assert np.array_equal(pp[b].cpu().numpy(), pp_o) and np.array_equal(gp[b].cpu().numpy(), gp_o)
                ev_o.add_image(pred3[b].copy(), gt3[b])
        ev_b.add_images(pt, gtt)
        rb, rs = ev_b.evaluate(), ev_s.evaluate()
        for k in ("pq", "sq", "rq", "tp", "fp", "fn", "iou_sum"):
            assert rb[k] == rs[k], k
        if pred3.shape[0] <= 2:
            ro = ev_o.evaluate()
            for k in ("pq", "sq", "rq", "tp", "fp", "fn", "iou_sum"):
                assert rb[k] == ro[k], k
        assert rb["per_class"] == rs["per_class"]


def test_joint_hist_batch_windows():
    """Overlapping windows (stride < n_per_table) and a table that has to grow."""
    from video_latent_diffusion_panoptic_segmentation_b200 import ops
    rng = np.random.default_rng(5)
    a = rng.integers(-1, 3000, size=(5, 64, 96)).astype(np.int32)
    b = rng.integers(0, 7, size=(5, 64, 96)).astype(np.int32)
    at, bt = torch.from_numpy(a).to(DEV), torch.from_numpy(b).to(DEV)
    hw = 64 * 96
    for k in (1, 2, 3):
        got = ops.joint_hist_batch(at, bt, 5 - k + 1, k * hw, hw, capacity=256)
        for w, (ga, gb, gc) in enumerate(got):
            key = a[w:w + k].astype(np.int64).ravel() * 16 + b[w:w + k].ravel()
            u, c = np.unique(key, return_counts=True)
            assert np.array_equal(ga * 16 + gb, u) and np.array_equal(gc, c)
