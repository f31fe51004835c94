"""Streaming sampler: per-image timesteps through the UNet and the DDIM, DPM-Solver++ and UniPC updates, and
TrainerDiffusion.sample_stream, which admits frames as slots free up.

On the CPU: the slot bookkeeping (stream_schedule) with a fake step, the noise rule and the refused modes. On the GPU,
every check is bit for bit against the existing batch path:
  the per-image UNet plan     : image b equals the uniform plan at t_b, with the same GEMM configuration per launch
  the *_rows update kernels   : image b's slice equals the existing kernel run at that image's row
  sample_stream               : every frame's final latents (and panoptic ids) equal sample()'s for a batch of the
                                same size that holds the frame at its slot with the same noise
"""
import random

import pytest
import torch

from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.schedulers import (
    DDIMNoiseScheduler, DPMSolverMultistepScheduler, UniPCMultistepScheduler)
from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.trainers import TrainerDiffusion
from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.trainers.trainers_ldm_cond import (
    stream_noise, stream_schedule)

KW = dict(num_train_timesteps=1000, beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear")
DDIM_KW = dict(KW, clip_sample=False, set_alpha_to_one=False, steps_offset=1, prediction_type="epsilon", weight="none")
DEV = "cuda"


# ---------------------------------------------------------------------------------------------------------- CPU
def _run_schedule(frames, N, B):
    """Drive stream_schedule with a fake step that records, per frame, the steps it ran; returns (steps per frame,
    admission order, finishing order, slot per frame)."""
    ran, admitted_order, finished_order, slot_of = {}, [], [], {}
    for admitted, steps, finished in stream_schedule(frames, N, B):
        for s, fid in admitted:
            assert steps[s] == 0 and fid not in ran
            admitted_order.append(fid)
            slot_of[fid] = s
            ran[fid] = []
        occupied = {slot_of[f]: f for f in ran if len(ran[f]) < N}
        assert sorted(occupied) == [s for s in range(B) if steps[s] is not None]
        for s, f in occupied.items():
            ran[f].append(steps[s])                              # the fake step
        for s, fid in finished:
            assert steps[s] == N - 1 and occupied.get(s) == fid  # never an empty slot
            finished_order.append(fid)
    return ran, admitted_order, finished_order, slot_of


@pytest.mark.parametrize("n_frames,B,N", [(11, 4, 3), (3, 8, 5), (1, 1, 1), (17, 2, 4), (8, 8, 1)],
                         ids=["11x4", "shorter-than-B", "single", "17x2", "N=1"])
def test_schedule_runs_every_frame_through_every_step_in_arrival_order(n_frames, B, N):
    ran, adm, fin, _ = _run_schedule(list(range(n_frames)), N, B)
    assert adm == list(range(n_frames))
    assert fin == list(range(n_frames))                # one N for all: frames finish in arrival order
    assert all(ran[f] == list(range(N)) for f in range(n_frames)), ran


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_schedule_with_irregular_arrivals(seed):
    """None items (nothing has arrived yet) leave free slots empty; every frame still runs steps 0..N-1 in order."""
    rng = random.Random(seed)
    frames = []
    for f in range(13):
        frames += [None] * rng.choice([0, 0, 1, 3])
        frames.append(f)
    frames += [None, None]
    ran, adm, fin, _ = _run_schedule(frames, 4, 3)
    assert adm == list(range(13)) and sorted(fin) == list(range(13))
    assert all(ran[f] == [0, 1, 2, 3] for f in range(13))


def test_schedule_admits_when_a_slot_frees_up():
    """A frame that finishes at forward k frees its slot for the next frame at forward k + 1."""
    evs = list(stream_schedule(range(5), 2, 2))
    assert [e[1] for e in evs] == [[0, 0], [1, 1], [0, 0], [1, 1], [0, None], [1, None]]
    assert [[f for _, f in e[0]] for e in evs] == [[0, 1], [], [2, 3], [], [4], []]


def test_stream_noise_is_the_seed_plus_frame_draw():
    for f in (0, 3, 17):
        want = torch.randn((1, 4, 6, 10), generator=torch.Generator().manual_seed(100 + f))
        assert torch.equal(stream_noise(f, 100, (4, 6, 10)), want)


class _StubUNet:
    def __init__(self, cross):
        self.cross = cross

    def has_cross_attention(self):
        return self.cross


@pytest.mark.parametrize("mode", ["self_condition", "classifier-free guidance", "differs per frame", "clip_sample"])
def test_refused_modes_raise_naming_the_mode(mode):
    p, kw, sched = {}, {}, DDIMNoiseScheduler(**DDIM_KW)
    unet = _StubUNet(cross=False)
    if mode == "self_condition":
        p = {"train_kwargs": {"self_condition": True}}
    elif mode == "classifier-free guidance":
        kw = dict(text_encoder=object(), tokenizer=object())
    elif mode == "differs per frame":
        kw, unet = dict(image_descriptor_model=object()), _StubUNet(cross=True)
    else:
        sched = DDIMNoiseScheduler(**dict(DDIM_KW, clip_sample=True))
    tr = TrainerDiffusion(p=p, unet_model=unet, noise_scheduler=sched, args={"gpu": 0}, **kw)
    with pytest.raises(NotImplementedError, match=mode):
        tr.sample_stream([], 4)


# ---------------------------------------------------------------------------------------------------------- GPU
def _bits(t):
    return t.contiguous().view(torch.int32)


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
    return dict(unet=unet, vae=vae)


def _run_recording_configs(unet, st):
    """Run a plan eagerly launch by launch; returns the (block_n, pair, split_k) of every GEMM launch."""
    from video_latent_diffusion_panoptic_segmentation_b200 import ops
    cfgs = []
    for fn, a, k in st.plan:
        fn(*a, **k)
        if fn is ops.gemm:
            cfgs.append(ops.gemm_last_config())
    return cfgs


def _check_per_image_plan(unet, B, h, w, ts):
    x = torch.randn((B, 8, h, w), generator=torch.Generator().manual_seed(3)).to(DEV)
    got = unet(x, torch.tensor(ts, device=DEV)).sample                      # 1-D, B elements: the per-image plan
    st = unet._get_plan(B, h, w, 8, per_image_t=True)
    assert st.graph is not None and st.per_image_t
    for b, t in enumerate(ts):
        ref = unet(x, torch.tensor(t, device=DEV)).sample                   # uniform plan at t_b
        assert torch.equal(_bits(got[b]), _bits(ref[b])), (b, t)
    # the conv1 launches take rowbias instead of bias: every launch keeps the uniform plan's configuration
    uni = unet._get_plan(B, h, w, 8)
    cfg_rows, cfg_uni = _run_recording_configs(unet, st), _run_recording_configs(unet, uni)
    assert len(cfg_rows) == len(cfg_uni) and cfg_rows == cfg_uni
    # graph replay equals the same plan run eagerly
    st.timesteps.copy_(torch.tensor(ts))
    st.sample.copy_(x)
    unet._run_plan(st)
    eager = st.out.clone()
    st.graph.replay()
    assert torch.equal(_bits(eager), _bits(st.out)) and torch.equal(_bits(eager), _bits(got))


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(48, 156), (20, 36)], ids=["48x156", "tail"])
def test_unet_per_image_plan_equals_uniform_plan_per_image(models, shape):
    _check_per_image_plan(models["unet"], 4, *shape, [981, 641, 301, 1])


@pytest.mark.gpu
def test_unet_per_image_plan_with_learnable_object_queries():
    from oracle import unet_oracle as UNO
    from video_latent_diffusion_panoptic_segmentation_b200.ldmseg.models import UNet
    o_unet = UNO.build_unet(seed=6, cross_attention_dim=768, learnable_queries=(128, 768))
    unet = UNet(device=DEV)
    unet.load_state_dict(o_unet.state_dict())
    _check_per_image_plan(unet, 4, 16, 24, [901, 500, 499, 21])


def _sched(kind, N, order=2, disable=()):
    if kind == "ddim":
        s = DDIMNoiseScheduler(**DDIM_KW)
        s.set_timesteps_inference(N)
    elif kind == "dpm":
        s = DPMSolverMultistepScheduler(**KW, solver_order=order)
        s.set_timesteps(N)
    else:
        s = UniPCMultistepScheduler(**KW, solver_order=order, disable_corrector=list(disable))
        s.set_timesteps(N)
    return s


ROWS_CASES = [("ddim", 1, ()), ("dpm", 1, ()), ("dpm", 2, ()), ("unipc", 1, ()), ("unipc", 2, ()), ("unipc", 3, ()),
              ("unipc", 1, (1, 4)), ("unipc", 2, (1, 4)), ("unipc", 3, (1, 4))]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,order,disable", ROWS_CASES,
                         ids=[f"{k}{o}{'-disabled' if d else ''}" for k, o, d in ROWS_CASES])
@pytest.mark.parametrize("tail", [0, 2], ids=["n%4=0", "tail"])
@pytest.mark.parametrize("inplace", [False, True])
def test_rows_kernels_equal_the_existing_kernel_per_image(kind, order, disable, tail, inplace):
    """Four images at four different rows (a partial last image with `tail`): every output and state buffer of image
    b equals the existing single-row kernel run on image b's slice at row b."""
    from video_latent_diffusion_panoptic_segmentation_b200 import ops
    N, B, epi = 10, 4, 4 * 7 * 11
    n = B * epi - tail
    s = _sched(kind, N, order, disable)
    coef = s.coef_table(DEV)
    steps = [0, 6, 9, 3]                               # first-order, middle, last and corrected rows
    ts = s.timesteps.cpu().tolist()
    rows_host = [ts[i] for i in steps] if kind == "ddim" else steps
    rows = torch.tensor(rows_host, dtype=torch.int32, device=DEV)
    g = torch.Generator().manual_seed(7)
    r = lambda: torch.randn((n,), generator=g).to(DEV)  # noqa: E731
    eps, x = r(), r()
    nstate = {"ddim": 1, "dpm": 1, "unipc": 1 + order}[kind]
    state = [r() for _ in range(nstate)]
    ref_prev, ref_state = torch.empty_like(x), [torch.empty_like(t) for t in state]
    for b in range(B):
        sl = slice(b * epi, min((b + 1) * epi, n))
        e_b, x_b, st_b = eps[sl].clone(), x[sl].clone(), [t[sl].clone() for t in state]
        prev_b = x_b if inplace else torch.empty_like(x_b)
        idx = torch.tensor([rows_host[b]], dtype=torch.int32, device=DEV)
        if kind == "ddim":
            ops.ddim_step(e_b, x_b, coef, idx, prev_sample=prev_b, pred_x0=st_b[0])
        elif kind == "dpm":
            ops.dpmpp_step(e_b, x_b, coef, idx, prev_b, st_b[0])
        else:
            ops.unipc_step(e_b, x_b, coef, idx, prev_b, st_b[0], st_b[1:])
        ref_prev[sl] = prev_b
        for t, t_b in zip(ref_state, st_b):
            t[sl] = t_b
    prev = x if inplace else torch.empty_like(x)
    if kind == "ddim":
        ops.ddim_step_rows(eps, x, coef, rows, epi, prev_sample=prev, pred_x0=state[0])
    elif kind == "dpm":
        ops.dpmpp_step_rows(eps, x, coef, rows, epi, prev, state[0])
    else:
        ops.unipc_step_rows(eps, x, coef, rows, epi, prev, state[0], state[1:])
    assert torch.equal(_bits(prev), _bits(ref_prev))
    for k, (t, t_ref) in enumerate(zip(state, ref_state)):
        assert torch.equal(_bits(t), _bits(t_ref)), k


@pytest.mark.gpu
def test_time_embedding_rows_equal_the_single_vector_chain(models):
    """timestep_sinusoid_rows and gemv_rows (segment-major) row b equal the single-vector launches at t_b."""
    from video_latent_diffusion_panoptic_segmentation_b200 import ops
    unet = models["unet"]
    unet._get_plan(2, 16, 24, 8)
    P = unet._packed
    ts = [999, 500, 1, 0, 250]
    B = len(ts)
    tdev = torch.tensor(ts, dtype=torch.int64, device=DEV)
    sin = ops.timestep_sinusoid_rows(tdev, P["freqs"], torch.empty((B, 2 * P["freqs"].numel()), device=DEV))
    e1 = ops.gemv_rows(P["t1"][0], sin, torch.empty((B, P["t1"][0].shape[0]), device=DEV), P["t1"][1], None, True)
    offs = sorted(o for o, _ in P["temb_offs"].values()) + [P["temb_total"]]
    seg = torch.tensor(offs, dtype=torch.int32, device=DEV)
    rows = ops.gemv_rows(P["temb_w"], e1, torch.empty((B * P["temb_total"],), device=DEV), P["temb_b"],
                         P["temb_conv1_b"], False, seg_offs=seg)
    for b, t in enumerate(ts):
        s1 = ops.timestep_sinusoid(tdev, torch.tensor([b], dtype=torch.int32, device=DEV), P["freqs"],
                                   torch.empty((2 * P["freqs"].numel(),), device=DEV))
        assert torch.equal(_bits(s1), _bits(sin[b]))
        v1 = ops.gemv(P["t1"][0], s1, torch.empty((P["t1"][0].shape[0],), device=DEV), P["t1"][1], None, True)
        assert torch.equal(_bits(v1), _bits(e1[b]))
        full = ops.gemv(P["temb_w"], v1, torch.empty((P["temb_total"],), device=DEV), P["temb_b"], P["temb_conv1_b"])
        for lo, hi in zip(offs[:-1], offs[1:]):
            blk = rows[lo * B:hi * B].view(B, hi - lo)
            assert torch.equal(_bits(blk[b]), _bits(full[lo:hi])), (b, lo)


def _rgb_of(f, h, w):
    return 0.18215 * torch.randn((1, 4, h, w), generator=torch.Generator().manual_seed(5000 + f))


STREAM_CASES = [("ddim", 10, 1), ("dpm", 8, 2), ("unipc", 6, 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,N,order", STREAM_CASES, ids=["ddim10", "dpmpp2m8", "unipc2-6"])
def test_sample_stream_equals_the_batch_sampler(models, kind, N, order):
    B, h, w, n_frames, seed = 4, 16, 24, 11, 42
    arrivals = []
    for f in range(n_frames):                         # staggered: frames arrive between forwards
        arrivals += [None] * (f % 3 == 1) + [f]
    frames = [None if a is None else (a, _rgb_of(a, h, w).to(DEV), None) for a in arrivals]
    tr = TrainerDiffusion(p={"eval_kwargs": {"mask_th": 0.0, "count_th": 64, "overlap_th": 0.0}},
                          vae_semseg=models["vae"], unet_model=models["unet"], noise_scheduler=_sched(kind, N, order),
                          args={"gpu": 0})
    got = dict(tr.sample_stream(iter(frames), N, batch_size=B, seed=seed))
    assert sorted(got) == list(range(n_frames))
    # the reference: sample() on batches of B in which every frame sits at the slot it had in the stream
    _, _, _, slot_of = _run_schedule([None if a is None else a for a in arrivals], N, B)
    per_slot = [[f for f in range(n_frames) if slot_of[f] == s] for s in range(B)]
    ref = {}
    for k in range(max(len(p) for p in per_slot)):
        batch = [p[k] if k < len(p) else None for p in per_slot]
        rgb = torch.cat([_rgb_of(f, h, w) if f is not None else torch.zeros((1, 4, h, w)) for f in batch])
        noise = torch.cat([stream_noise(f, seed, (4, h, w)) if f is not None else torch.zeros((1, 4, h, w))
                           for f in batch])
        lat = tr.sample([""] * B, num_inference_steps=N, scheduler=_sched(kind, N, order), rgb_latents=rgb.to(DEV),
                        noise=noise)
        for s, f in enumerate(batch):
            if f is not None:
                ref[f] = lat[s:s + 1]
    for f in range(n_frames):
        assert torch.equal(_bits(got[f]), _bits(ref[f])), f
    # panoptic ids, decoded in batches of B in frame order
    for k in range(0, n_frames, B):
        fs = list(range(k, min(k + B, n_frames)))
        _, c_got, _ = tr.panoptic_ids(torch.cat([got[f] for f in fs]))
        _, c_ref, _ = tr.panoptic_ids(torch.cat([ref[f] for f in fs]))
        assert torch.equal(c_got, c_ref)
