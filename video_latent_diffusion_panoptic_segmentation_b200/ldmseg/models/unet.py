"""B200 host mirror of ``ldmseg/models/unet.py`` (reference ``class UNet(UNet2DConditionModel)``, :24-436).

Same call surface on the sampling path -- ``forward(sample, timestep, encoder_hidden_states, ...) -> UNetOutput``,
``modify_encoder``, ``remove_cross_attention``, ``freeze_layers``, ``load_state_dict`` with diffusers key names,
``.dtype/.device/.config.block_out_channels/.conv_in`` -- but every tensor op is a hand-written sm_100a kernel behind
the C ABI (ops.py). PyTorch only owns the device memory. There is no eager / CPU fallback.

Execution model: the first forward for a given (B, h, w) builds a static *plan* -- packed bf16 weights, an arena of
NHWC activation buffers with liveness-based reuse, and a flat list of kernel launches -- runs it once eagerly and then
captures it into a CUDA graph; later calls copy the inputs into the static buffers and replay the graph (the timestep
is read on the device, so one graph serves all DDIM steps and there is no host sync in the loop).
"""
import math
from types import SimpleNamespace

import torch

from .. import utils as U
from ... import _lib as L
from ... import ops

bf16, f32 = torch.bfloat16, torch.float32


class UNetOutput(U.OutputDict):
    """ldmseg/models/unet.py:20-21"""
    sample: torch.Tensor


SD14_CONFIG = dict(
    in_channels=4, out_channels=4, block_out_channels=(320, 640, 1280, 1280), layers_per_block=2,
    attention_head_dim=8,  # diffusers quirk: this is the NUMBER of heads
    norm_num_groups=32, norm_eps=1e-5, cross_attention_dim=768,
    down_block_types=("CrossAttnDownBlock2D", "CrossAttnDownBlock2D", "CrossAttnDownBlock2D", "DownBlock2D"),
    up_block_types=("UpBlock2D", "CrossAttnUpBlock2D", "CrossAttnUpBlock2D", "CrossAttnUpBlock2D"),
)


class _Arena:
    """Reusable device buffers keyed by byte size. The plan is built and executed in program order on one stream,
    so a buffer released at build time can safely back a later tensor."""

    def __init__(self, device):
        self.device = device
        self.free = {}
        self.total = 0

    def alloc(self, shape, dtype=bf16):
        n = int(math.prod(shape)) * torch.empty((), dtype=dtype).element_size()
        n = (n + 1023) // 1024 * 1024
        lst = self.free.get(n)
        if lst:
            raw = lst.pop()
        else:
            raw = torch.empty(n, dtype=torch.uint8, device=self.device)
            self.total += n
        t = raw.view(dtype)[: int(math.prod(shape))].view(shape)
        t._arena_raw = raw
        return t

    def release(self, t):
        raw = getattr(t, "_arena_raw", None)
        if raw is not None:
            self.free.setdefault(raw.numel(), []).append(raw)


class _ConvInProxy:
    """What callers read from ``unet.conv_in`` (unet.py:180-183,216-220): channel counts and fp32 weight/bias."""

    def __init__(self, weight, bias):
        self.weight, self.bias = weight, bias
        self.out_channels, self.in_channels = weight.shape[0], weight.shape[1]
        self.kernel_size, self.stride, self.padding = (3, 3), (1, 1), (1, 1)


class UNet:
    def __init__(self, device="cuda", **config):
        cfg = dict(SD14_CONFIG)
        cfg.update(config)
        self.config = SimpleNamespace(**cfg)
        self.device = torch.device(device)
        self.dtype = torch.float32  # the reference keeps fp32 parameters (main_ldm.py:169); compute here is bf16/fp32-acc
        self.compute_dtype = "bf16"
        self._sd = None          # fp32 CPU state dict (diffusers key names)
        self._packed = None      # device weights
        self._plans = {}
        self._cross_attention_removed = False
        self.encoder_hid_proj = None
        self.use_cuda_graph = True
        # BasicTransformerBlock's LayerNorms folded into the GEMMs around them (ldm_gemm_desc.ln_stats) instead of
        # ldm_layernorm passes. Built, parity-checked and measured (tools/bench_ln_fold.py, DESIGN.md 3): it removes
        # 0.54 ms of LayerNorm per forward but the QKV / GEGLU epilogues it lands in are issue-bound at K = 320 - 640
        # and pay 0.9 ms for it, so the default is the separate pass.
        self.ln_fold = False
        # Upsample2D as four sub-pixel 2x2 convolutions (ldm_gemm_desc.up2) from this many low-resolution rows (B*H*W) on;
        # below, the per-class GEMMs are too small and the nearest-upsample pass + one 3x3 convolution is faster
        self.up2_min_rows = 1800
        self.training = False

    # ------------------------------------------------------------------ construction (main_ldm.py:147-169)
    @classmethod
    def from_pretrained(cls, path=None, subfolder="unet", device="cuda", state_dict=None, **config):
        """The reference loads SD-1.4 weights from disk through diffusers; here the caller passes the diffusers-keyed
        ``state_dict`` (e.g. from a checkpoint's ``data['unet']``) or random-inits through the oracle builder."""
        net = cls(device=device, **config)
        if state_dict is not None:
            net.load_state_dict(state_dict)
        elif path is not None:
            data = torch.load(path, map_location="cpu")
            net.load_state_dict(data["unet"] if "unet" in data else data)
        return net

    def load_state_dict(self, sd, strict=True):
        sd = {k.replace("module.", ""): v.detach().to("cpu", f32) for k, v in sd.items()}
        if any(".attn2." in k for k in sd) and self._cross_attention_removed is False:
            # cross-attention weights present: they are dropped by remove_cross_attention (unet.py:83-105)
            pass
        self._sd = sd
        self._packed = None
        self._plans = {}
        w = sd["conv_in.weight"]
        self.conv_in = _ConvInProxy(w, sd["conv_in.bias"])
        return "<All keys matched successfully>"

    def state_dict(self):
        return dict(self._sd)

    def remove_cross_attention(self):
        """unet.py:83-105: attn2/norm2 of every transformer block are dropped; only self-attention remains."""
        if self._sd is not None:
            self._sd = {k: v for k, v in self._sd.items() if ".attn2." not in k and ".norm2." not in k
                        or ".resnets." in k}
        self._cross_attention_removed = True
        self._packed = None
        self._plans = {}

    def modify_encoder(self, in_channels=4, init_mode_seg="copy", init_mode_image="copy", cond_channels=0,
                       init_mode_cond="zero", separate_conv=False, separate_encoder=False, add_adaptor=False,
                       init_mode_adaptor="random"):
        """unet.py:124-233 (in_channels == 8 branch): build the (8+cond)-channel conv_in from the 4-channel one."""
        assert in_channels in [4, 8], "in_channels must be 4 or 8"
        if separate_conv or separate_encoder:
            raise NotImplementedError("separate_conv / separate_encoder are not on the default sampling path")
        if in_channels != 8:
            return
        old_w, old_b = self._sd["conv_in.weight"], self._sd["conv_in.bias"]
        cout = old_w.shape[0]
        new = torch.nn.Conv2d(in_channels + cond_channels, cout, 3, padding=1)
        new_w = new.weight.detach().clone()
        for sl, mode in ((slice(0, 4), init_mode_seg), (slice(4, 8), init_mode_image)):
            if mode in ("copy", "div"):  # the reference's "/ 2." acts on a discarded temporary (unet.py:188,202)
                new_w[:, sl] = old_w
            elif mode == "mean":
                new_w[:, sl] = old_w.mean(dim=1, keepdim=True).repeat(1, 4, 1, 1)
            elif mode == "zero":
                new_w[:, sl] = 0
            elif mode != "random":
                raise NotImplementedError(f"init_mode {mode} not implemented")
        if cond_channels > 0:
            if init_mode_cond == "zero":
                new_w[:, 8:] = 0
            elif init_mode_cond != "random":
                raise NotImplementedError(f"init_mode cond {init_mode_cond} not implemented")
        assert new_w.shape == torch.Size([cout, 8 + cond_channels, 3, 3])
        self._sd["conv_in.weight"] = new_w
        self._sd["conv_in.bias"] = old_b.clone()
        self._sd["new_conv.weight"] = self._sd["conv_in.weight"]  # alias kept by the reference (unet.py:182,233)
        self._sd["new_conv.bias"] = self._sd["conv_in.bias"]
        self.conv_in = _ConvInProxy(new_w, self._sd["conv_in.bias"])
        self._packed = None
        self._plans = {}

    def modify_encoder_hidden_state_proj(self, in_channels, out_channels):
        """unet.py:122-123: a fresh nn.Linear in front of the cross-attention context (CLIP image features 1024 -> 768)."""
        lin = torch.nn.Linear(in_channels, out_channels)
        self._sd["encoder_hid_proj.weight"] = lin.weight.detach().clone()
        self._sd["encoder_hid_proj.bias"] = lin.bias.detach().clone()
        self.encoder_hid_proj = lin
        self._packed, self._plans = None, {}

    def define_learnable_embeddings(self, num_queries, dim):
        """image_descriptors == 'learnable' (descriptors.py:89-91): an nn.Embedding whose weight is the context."""
        emb = torch.nn.Embedding(num_queries, dim)
        self._sd["object_queries.weight"] = emb.weight.detach().clone()
        self.object_queries = emb
        self._packed, self._plans = None, {}

    def has_cross_attention(self):
        """True when the transformer blocks keep norm2 / attn2 (SD weights loaded and remove_cross_attention() not called)."""
        return (not self._cross_attention_removed) and any(".attn2." in k for k in (self._sd or {}))

    def freeze_layers(self, layers=("norm", "time_embedding")):
        return None  # inference-only mirror: nothing is trainable

    def to(self, *args, **kwargs):
        for a in args:
            if isinstance(a, (str, torch.device, int)):
                self.device = torch.device(a if not isinstance(a, int) else f"cuda:{a}")
        return self

    def eval(self):
        return self

    def parameters(self):
        return iter(self._sd.values())

    # ------------------------------------------------------------------ weight packing
    def _pack(self):
        sd, dev = self._sd, self.device
        P = {}
        P["cross"] = (not self._cross_attention_removed) and any(".attn2." in k for k in sd)

        def dv(t, dtype=f32):
            return t.to(dev, dtype).contiguous()

        def conv3(name):
            w = sd[name + ".weight"]
            return dv(w.permute(0, 2, 3, 1).reshape(w.shape[0], -1), bf16), dv(sd[name + ".bias"])

        def lin(name, bias=True):
            w = sd[name + ".weight"]
            return dv(w.reshape(w.shape[0], -1), bf16), (dv(sd[name + ".bias"]) if bias else None)

        def norm(name):
            return dv(sd[name + ".weight"]), dv(sd[name + ".bias"])

        P["conv_in"] = (dv(ops.pack_small_cin_weight(sd["conv_in.weight"])), dv(sd["conv_in.bias"]))
        wo, bo = sd["conv_out.weight"], sd["conv_out.bias"]  # [4, C, 3, 3] -> tap-major rows, zero-padded to 8 outputs
        npad = (wo.shape[0] + 7) // 8 * 8
        wop = torch.zeros((npad, 9 * wo.shape[1]))
        wop[: wo.shape[0]] = wo.permute(0, 2, 3, 1).reshape(wo.shape[0], -1)
        bop = torch.zeros((npad,))
        bop[: wo.shape[0]] = bo
        P["conv_out"] = (dv(wop, bf16), dv(bop))
        P["conv_norm_out"] = norm("conv_norm_out")
        P["t1"], P["t2"] = lin("time_embedding.linear_1"), lin("time_embedding.linear_2")
        half = sd["time_embedding.linear_1.weight"].shape[1] // 2
        exponent = -math.log(10000) * torch.arange(0, half, dtype=f32)
        P["freqs"] = dv(torch.exp(exponent / half))

        res_names = [k[: -len(".norm1.weight")] for k in sd if k.endswith(".norm1.weight") and ".resnets." in k]
        temb_w, temb_b, conv1_b, offs = [], [], [], {}
        o = 0
        for r in res_names:
            w = sd[r + ".time_emb_proj.weight"]
            temb_w.append(w); temb_b.append(sd[r + ".time_emb_proj.bias"]); conv1_b.append(sd[r + ".conv1.bias"])
            offs[r] = (o, w.shape[0])
            o += w.shape[0]
            P[r + ".norm1"], P[r + ".norm2"] = norm(r + ".norm1"), norm(r + ".norm2")
            P[r + ".conv1"], P[r + ".conv2"] = conv3(r + ".conv1"), conv3(r + ".conv2")
            if r + ".conv_shortcut.weight" in sd:
                P[r + ".conv_shortcut"] = lin(r + ".conv_shortcut")
        P["temb_w"] = dv(torch.cat(temb_w, 0), bf16)
        P["temb_b"], P["temb_conv1_b"] = dv(torch.cat(temb_b, 0)), dv(torch.cat(conv1_b, 0))
        P["temb_offs"], P["temb_total"] = offs, o

        attn_names = [k[: -len(".proj_in.weight")] for k in sd if k.endswith(".proj_in.weight")]
        for a in attn_names:
            tb = a + ".transformer_blocks.0"
            P[a + ".norm"] = norm(a + ".norm")
            P[a + ".proj_in"], P[a + ".proj_out"] = lin(a + ".proj_in"), lin(a + ".proj_out")
            P[tb + ".norm1"], P[tb + ".norm3"] = norm(tb + ".norm1"), norm(tb + ".norm3")
            wqkv = torch.cat([sd[tb + ".attn1.to_q.weight"], sd[tb + ".attn1.to_k.weight"],
                              sd[tb + ".attn1.to_v.weight"]], 0)
            if not self.ln_fold:
                P[tb + ".qkv"] = dv(wqkv, bf16)

            def folded(w, b, ln):
                """(gamma o W in bf16, b + W beta, row sums of the rounded gamma o W): the Linear behind LayerNorm `ln`
                in the form the GEMM epilogue normalises itself (ldm_gemm_desc.ln_stats)."""
                w2, b2, cs = ops.fold_layernorm(w.float(), b, sd[ln + ".weight"].float(), sd[ln + ".bias"].float())
                return dv(w2, bf16), dv(b2), dv(cs)

            if self.ln_fold:
                P[tb + ".qkv_ln"] = folded(wqkv, None, tb + ".norm1")
            P[tb + ".to_out"] = lin(tb + ".attn1.to_out.0")
            w1, b1 = sd[tb + ".ff.net.0.proj.weight"], sd[tb + ".ff.net.0.proj.bias"]
            inner = w1.shape[0] // 2
            idx = torch.arange(inner).view(-1, 16)
            perm = torch.cat([idx, idx + inner], dim=1).reshape(-1)  # 16 value rows, then their 16 gate rows
            if not self.ln_fold:
                P[tb + ".ff1"] = (dv(w1[perm], bf16), dv(b1[perm]))
            else:
                P[tb + ".ff1_ln"] = folded(w1[perm], b1[perm], tb + ".norm3")
            P[tb + ".ff2"] = lin(tb + ".ff.net.2")
            if P["cross"]:  # BasicTransformerBlock.norm2 / attn2 against encoder_hidden_states (SURVEY 8f rank 4)
                P[tb + ".norm2"] = norm(tb + ".norm2")
                if not self.ln_fold:
                    P[tb + ".q2"] = dv(sd[tb + ".attn2.to_q.weight"], bf16)
                else:
                    P[tb + ".q2_ln"] = folded(sd[tb + ".attn2.to_q.weight"], None, tb + ".norm2")
                P[tb + ".kv2"] = dv(torch.cat([sd[tb + ".attn2.to_k.weight"], sd[tb + ".attn2.to_v.weight"]], 0), bf16)
                P[tb + ".to_out2"] = lin(tb + ".attn2.to_out.0")
        if P["cross"]:
            P["ctx_dim"] = sd[attn_names[0] + ".transformer_blocks.0.attn2.to_k.weight"].shape[1]
            if "encoder_hid_proj.weight" in sd:    # unet.py:122-123,319-320
                P["hid_proj"] = lin("encoder_hid_proj")
            if "object_queries.weight" in sd:      # unet.py:322-323 (image_descriptors == 'learnable')
                P["object_queries"] = dv(sd["object_queries.weight"], bf16)
        for k in sd:
            if k.endswith("samplers.0.conv.weight"):
                P[k[: -len(".weight")]] = conv3(k[: -len(".weight")])
                if ".upsamplers." in k:  # nearest x2 + conv3x3 as four 2x2 convolutions (ldm_gemm_desc.up2)
                    w4, b4 = ops.fold_upsample_conv3x3(sd[k].permute(0, 2, 3, 1), sd[k[: -len(".weight")] + ".bias"])
                    P[k[: -len(".weight")] + ".up2"] = (dv(w4, bf16), dv(b4))
        self._packed = P

    # ------------------------------------------------------------------ plan
    def _build_plan(self, B, h, w, cin, ctx_len=0, per_image_t=False):
        if self._packed is None:
            self._pack()
        P, cfg, dev = self._packed, self.config, self.device
        cross = P["cross"]
        if cross and ctx_len <= 0:
            raise L.LdmError("this UNet keeps its cross-attention layers: pass encoder_hidden_states (or call "
                             "define_learnable_embeddings / remove_cross_attention as tools/main_ldm.py does)")
        ch = list(cfg.block_out_channels)
        heads, groups, eps = cfg.attention_head_dim, cfg.norm_num_groups, cfg.norm_eps
        nres = cfg.layers_per_block
        arena = _Arena(dev)
        plan = []
        st = SimpleNamespace()
        st.in_parts = None
        st.sample = torch.zeros((B, cin, h, w), dtype=f32, device=dev)     # static input (concatenated form)
        st.per_image_t = per_image_t
        if per_image_t:
            st.timesteps = torch.zeros((B,), dtype=torch.int64, device=dev)  # static timestep of every image
        else:
            st.timestep = torch.zeros((1,), dtype=torch.int64, device=dev)   # static timestep
        st.out = torch.empty((B, cfg.out_channels, h, w), dtype=f32, device=dev)
        st.gn_stats = ops.gn_scratch(B, groups, dev)
        temb_dim = P["t1"][0].shape[0]
        st.sinus = torch.empty((2 * P["freqs"].numel(),), dtype=f32, device=dev)
        st.emb1 = torch.empty((temb_dim,), dtype=f32, device=dev)
        st.emb_silu = torch.empty((temb_dim,), dtype=f32, device=dev)
        st.temb_bias = torch.empty((P["temb_total"],), dtype=f32, device=dev)
        qkv_cache = {}
        ln_stats_cache = {}  # per-row LayerNorm moments [C/32, M, 2], one buffer per level (producer -> consumer in stream order)
        ctx_plan = []  # launches that depend only on the context: run when it changes, not once per DDIM step
        st.ctx_len, st.context_in, st.context = ctx_len, None, None
        if cross:
            in_dim = P["hid_proj"][0].shape[1] if "hid_proj" in P else P["ctx_dim"]
            st.context_in = torch.zeros((B * ctx_len, in_dim), dtype=bf16, device=dev)
            if "hid_proj" in P:
                st.context = torch.empty((B * ctx_len, P["ctx_dim"]), dtype=bf16, device=dev)
                ctx_plan.append((ops.gemm, (st.context_in, P["hid_proj"][0], st.context), dict(bias=P["hid_proj"][1])))
            else:
                st.context = st.context_in

        def add(fn, *a, **k):
            plan.append((fn, a, k))

        # 1. time embedding chain (unet.py:301-307) -> per-resnet conv1 biases (conv1.bias + time_emb_proj(silu(emb)))
        if per_image_t:
            # one embedding per image; the last GEMV writes segment-major [resnet][B][n_r], so every conv1 reads a
            # contiguous [B, n_r] rowbias block. Each row's arithmetic is that of the single-vector chain.
            st.sinus = torch.empty((B, 2 * P["freqs"].numel()), dtype=f32, device=dev)
            st.emb1 = torch.empty((B, temb_dim), dtype=f32, device=dev)
            st.emb_silu = torch.empty((B, temb_dim), dtype=f32, device=dev)
            st.temb_rows = torch.empty((B * P["temb_total"],), dtype=f32, device=dev)
            st.temb_seg_offs = torch.tensor(sorted(o for o, _ in P["temb_offs"].values()) + [P["temb_total"]],
                                            dtype=torch.int32, device=dev)
            add(ops.timestep_sinusoid_rows, st.timesteps, P["freqs"], st.sinus)
            add(ops.gemv_rows, P["t1"][0], st.sinus, st.emb1, P["t1"][1], None, True)
            add(ops.gemv_rows, P["t2"][0], st.emb1, st.emb_silu, P["t2"][1], None, True)
            add(ops.gemv_rows, P["temb_w"], st.emb_silu, st.temb_rows, P["temb_b"], P["temb_conv1_b"], False,
                seg_offs=st.temb_seg_offs)
        else:
            add(ops.timestep_sinusoid, st.timestep, None, P["freqs"], st.sinus)
            add(ops.gemv, P["t1"][0], st.sinus, st.emb1, P["t1"][1], None, True)
            add(ops.gemv, P["t2"][0], st.emb1, st.emb_silu, P["t2"][1], None, True)
            add(ops.gemv, P["temb_w"], st.emb_silu, st.temb_bias, P["temb_b"], P["temb_conv1_b"], False)

        def resnet(name, xa, xb, H, W):
            c1 = xa.shape[-1]
            c2 = xb.shape[-1] if xb is not None else 0
            cout = P[name + ".conv1"][0].shape[0]
            t0 = arena.alloc((B, H, W, c1 + c2))
            add(ops.groupnorm, xa, *P[name + ".norm1"], t0, st.gn_stats, x2=xb, groups=groups, eps=eps, silu=True)
            o, n = P["temb_offs"][name]
            t1 = arena.alloc((B, H, W, cout))
            if per_image_t:  # the epilogue adds 0 + rowbias: exactly the uniform plan's bias for that image's t
                tb_ = dict(rowbias=st.temb_rows[o * B:(o + n) * B].view(B, n))
            else:
                tb_ = dict(bias=st.temb_bias[o:o + n])
            add(ops.gemm, t0, P[name + ".conv1"][0], t1, taps=9, **tb_)
            arena.release(t0)
            t2 = arena.alloc((B, H, W, cout))
            add(ops.groupnorm, t1, *P[name + ".norm2"], t2, st.gn_stats, groups=groups, eps=eps, silu=True)
            arena.release(t1)
            if name + ".conv_shortcut" in P:
                sc = arena.alloc((B, H, W, cout))
                add(ops.gemm, xa, P[name + ".conv_shortcut"][0], sc, a2=xb, taps=1, bias=P[name + ".conv_shortcut"][1])
            else:
                assert xb is None and c1 == cout
                sc = xa
            out = arena.alloc((B, H, W, cout))
            add(ops.gemm, t2, P[name + ".conv2"][0], out, taps=9, bias=P[name + ".conv2"][1],
                residual=sc.view(B * H * W, cout))
            arena.release(t2)
            if sc is not xa:
                arena.release(sc)
            return out

        def transformer(name, x, H, W):
            C = x.shape[-1]
            M, seq, d = B * H * W, H * W, C // heads
            tb = name + ".transformer_blocks.0"
            key = (seq, d)
            if key not in qkv_cache:  # zero-padded head-split buffers, shared by all layers of this level
                qkv_cache[key] = ops.alloc_qkv(B, heads, seq, d, dev)
            qkv = qkv_cache[key]
            t0 = arena.alloc((B, H, W, C))
            add(ops.groupnorm, x, *P[name + ".norm"], t0, st.gn_stats, groups=groups, eps=1e-6, silu=False)
            hid = arena.alloc((M, C))
            # LayerNorm folded into the GEMMs on both sides of it (ops.gemm row_stats / ln_fold): the GEMM that writes
            # the residual stream also writes its per-row moments, the QKV / GEGLU GEMM normalises in its epilogue
            fold = self.ln_fold
            if fold and (M, C) not in ln_stats_cache:
                ln_stats_cache[(M, C)] = torch.empty(((C + 31) // 32, M, 2), dtype=f32, device=dev)
            rs = ln_stats_cache[(M, C)] if fold else None
            add(ops.gemm, t0.view(M, C), P[name + ".proj_in"][0], hid, bias=P[name + ".proj_in"][1], row_stats=rs)
            arena.release(t0)
            t1 = arena.alloc((M, C))
            if fold:
                wq, bq, csq = P[tb + ".qkv_ln"]
                add(ops.gemm, hid, wq, None, bias=bq, flags=L.LDM_GEMM_QKV_SPLIT, qkv=qkv, ln_fold=(rs, csq, 1e-5))
            else:
                add(ops.layernorm, hid, *P[tb + ".norm1"], t1, 1e-5)
                add(ops.gemm, t1, P[tb + ".qkv"], None, flags=L.LDM_GEMM_QKV_SPLIT, qkv=qkv)
            add(ops.flash_attn, qkv["q"], qkv["k"], qkv["vt"], t1, B=B, heads=heads, seq=seq, head_dim=d,
                dpad=qkv["dpad"], seq_pad=qkv["seq_pad"], scale=d ** -0.5)
            h2 = arena.alloc((M, C))
            add(ops.gemm, t1, P[tb + ".to_out"][0], h2, bias=P[tb + ".to_out"][1], residual=hid, row_stats=rs)
            arena.release(t1)
            arena.release(hid)
            if cross:
                # attn2: q from the tokens, k / v from the context (projected once per context into per-layer buffers)
                kv = ops.alloc_kv(B, heads, ctx_len, d, dev)
                ctx_plan.append((ops.gemm, (st.context, P[tb + ".kv2"], None),
                                 dict(flags=L.LDM_GEMM_QKV_SPLIT, qkv=dict(kv, part0=1))))
                t1 = arena.alloc((M, C))
                q_only = dict(q=qkv["q"], heads=heads, head_dim=d, dpad=qkv["dpad"], seq=seq, seq_pad=qkv["seq_pad"])
                if fold:
                    wq2, bq2, csq2 = P[tb + ".q2_ln"]
                    add(ops.gemm, h2, wq2, None, bias=bq2, flags=L.LDM_GEMM_QKV_SPLIT, qkv=q_only, ln_fold=(rs, csq2, 1e-5))
                else:
                    add(ops.layernorm, h2, *P[tb + ".norm2"], t1, 1e-5)
                    add(ops.gemm, t1, P[tb + ".q2"], None, flags=L.LDM_GEMM_QKV_SPLIT, qkv=q_only)
                add(ops.flash_attn, qkv["q"], kv["k"], kv["vt"], t1, B=B, heads=heads, seq=seq, head_dim=d,
                    dpad=kv["dpad"], seq_pad=kv["seq_pad"], scale=d ** -0.5, kv_seq=ctx_len)
                h2b = arena.alloc((M, C))
                add(ops.gemm, t1, P[tb + ".to_out2"][0], h2b, bias=P[tb + ".to_out2"][1], residual=h2, row_stats=rs)
                arena.release(t1)
                arena.release(h2)
                h2 = h2b
            g = arena.alloc((M, 4 * C))
            if fold:
                wf, bf_, csf = P[tb + ".ff1_ln"]
                add(ops.gemm, h2, wf, g, bias=bf_, flags=L.LDM_GEMM_GEGLU, ln_fold=(rs, csf, 1e-5))
            else:
                t2 = arena.alloc((M, C))
                add(ops.layernorm, h2, *P[tb + ".norm3"], t2, 1e-5)
                add(ops.gemm, t2, P[tb + ".ff1"][0], g, bias=P[tb + ".ff1"][1], flags=L.LDM_GEMM_GEGLU)
                arena.release(t2)
            h3 = arena.alloc((M, C))
            add(ops.gemm, g, P[tb + ".ff2"][0], h3, bias=P[tb + ".ff2"][1], residual=h2)
            arena.release(g)
            arena.release(h2)
            out = arena.alloc((B, H, W, C))
            add(ops.gemm, h3, P[name + ".proj_out"][0], out.view(M, C), bias=P[name + ".proj_out"][1],
                residual=x.view(M, C))
            arena.release(h3)
            return out

        # 2. conv_in fused with the concat + cast (trainers_ldm_cond.py:1131-1141, unet.py:357)
        x = arena.alloc((B, h, w, ch[0]))
        st.conv_in_slot = len(plan)
        add(ops.conv3x3_small_cin, [st.sample], P["conv_in"][0], P["conv_in"][1], x, 1.0)
        st.conv_in_out = x
        H, W = h, w
        skips = [(x, H, W)]
        keep = {id(x)}

        # 3. down blocks (unet.py:360-373)
        for i, co in enumerate(ch):
            has_attn = cfg.down_block_types[i].startswith("CrossAttn")
            for j in range(nres):
                y = resnet(f"down_blocks.{i}.resnets.{j}", x, None, H, W)
                if id(x) not in keep:
                    arena.release(x)
                x = y
                if has_attn:
                    y = transformer(f"down_blocks.{i}.attentions.{j}", x, H, W)
                    arena.release(x)
                    x = y
                skips.append((x, H, W))
                keep.add(id(x))
            if i < len(ch) - 1:
                # Downsample2D: Conv2d(3x3, stride 2, padding 1) as an implicit GEMM -- the A tensor map steps by two
                # pixels (ldm_gemm_desc.a_stride), no im2col buffer (it was 9x the input, written and read back)
                oh, ow = (H - 1) // 2 + 1, (W - 1) // 2 + 1
                y = arena.alloc((B, oh, ow, co))
                wd_, bd_ = P[f"down_blocks.{i}.downsamplers.0.conv"]
                add(ops.gemm, x, wd_, y, taps=9, bias=bd_, a_stride=2, a_pad=1)
                x, H, W = y, oh, ow
                skips.append((x, H, W))
                keep.add(id(x))

        # 4. mid block (unet.py:388-395)
        y = resnet("mid_block.resnets.0", x, None, H, W)
        x = y  # previous x is a skip
        y = transformer("mid_block.attentions.0", x, H, W)
        arena.release(x)
        x = y
        y = resnet("mid_block.resnets.1", x, None, H, W)
        arena.release(x)
        x = y

        # 5. up blocks (unet.py:401-425); Upsample2D takes the next skip's size (SURVEY fact 7)
        n_up = len(ch) - 1
        for i in range(len(ch)):
            has_attn = cfg.up_block_types[i].startswith("CrossAttn")
            for j in range(nres + 1):
                sk, sH, sW = skips.pop()
                assert (sH, sW) == (H, W), f"skip {sH}x{sW} does not match {H}x{W}"
                y = resnet(f"up_blocks.{i}.resnets.{j}", x, sk, H, W)
                arena.release(x)
                arena.release(sk)
                x = y
                if has_attn:
                    y = transformer(f"up_blocks.{i}.attentions.{j}", x, H, W)
                    arena.release(x)
                    x = y
            if i < n_up:
                oh, ow = skips[-1][1], skips[-1][2]
                cu = x.shape[-1]
                y = arena.alloc((B, oh, ow, cu))
                if (oh, ow) == (2 * H, 2 * W) and B * H * W >= self.up2_min_rows:
                    # Upsample2D: the up-sampled copy is never made -- four 2x2 convolutions of the low-resolution map
                    # (one per output parity), 4/9 of the multiply-adds, stored through a map that steps by two pixels
                    wu4, bu4 = P[f"up_blocks.{i}.upsamplers.0.conv.up2"]
                    add(ops.gemm, x, wu4, y, taps=4, bias=bu4, up2=True)
                    arena.release(x)
                else:  # odd target size (20 -> 39 columns), or too few rows to fill the SMs four times over
                    up = arena.alloc((B, oh, ow, cu))
                    add(ops.upsample_nearest, x, up)
                    arena.release(x)
                    wu, bu = P[f"up_blocks.{i}.upsamplers.0.conv"]
                    add(ops.gemm, up, wu, y, taps=9, bias=bu)
                    arena.release(up)
                x, H, W = y, oh, ow

        # 6. conv_norm_out + SiLU + conv_out (unet.py:428-431) -> fp32 NCHW
        t = arena.alloc((B, H, W, ch[0]))
        add(ops.groupnorm, x, *P["conv_norm_out"], t, st.gn_stats, groups=groups, eps=eps, silu=True)
        add(ops.gemm, t, P["conv_out"][0], st.out, taps=9, bias=P["conv_out"][1], flags=L.LDM_GEMM_OUT_NCHW_F32,
            block_n=32, n_store=cfg.out_channels)
        st.plan, st.arena_bytes, st.graph = plan, arena.total, None
        st.ctx_plan = ctx_plan
        if cross and "object_queries" in P:  # the context is a parameter: project it now, once
            st.context_in.view(B, ctx_len, -1).copy_(P["object_queries"].unsqueeze(0).expand(B, -1, -1))
            self._run_ctx_plan(st)
        st.launches_per_forward = None
        return st

    def _run_plan(self, st):
        for fn, a, k in st.plan:
            fn(*a, **k)

    def _run_ctx_plan(self, st):
        for fn, a, k in st.ctx_plan:
            fn(*a, **k)

    def set_context(self, st, encoder_hidden_states):
        """encoder_hidden_states [B, L, dim] -> the plan's static context; (re)projects k / v of every attn2 layer
        (and encoder_hid_proj, unet.py:319-320). The UNet graph reads those buffers, so one call serves all steps."""
        B = st.sample.shape[0]
        e = encoder_hidden_states
        if e.dim() != 3 or e.shape[0] != B or e.shape[1] != st.ctx_len or e.shape[2] != st.context_in.shape[1]:
            raise ValueError(f"encoder_hidden_states {tuple(e.shape)} does not match (B={B}, L={st.ctx_len}, "
                             f"dim={st.context_in.shape[1]})")
        st.context_in.view(B, st.ctx_len, -1).copy_(e)
        self._run_ctx_plan(st)

    def _get_plan(self, B, h, w, cin, parts=None, ctx_len=None, per_image_t=False):
        """parts: optional list of static f32 NCHW [B,4,h,w] buffers (x_t, rgb_latents[, condition]) that conv_in
        reads directly -- the sampler's fused concat (trainers_ldm_cond.py:1134-1141). ctx_len: tokens of the
        cross-attention context (default: the learnable object queries' count, or 0 without cross-attention).
        per_image_t: a plan whose static input is one timestep per image (`st.timesteps` int64 [B]) instead of one
        for the batch (`st.timestep`); it has its own cache entry and CUDA graph."""
        if self._packed is None:
            self._pack()
        if ctx_len is None:
            oq = self._packed.get("object_queries")
            ctx_len = oq.shape[0] if oq is not None else 0
        if not self._packed["cross"]:
            ctx_len = 0
        key = (B, h, w, cin, ctx_len, None if parts is None else tuple(t.data_ptr() for t in parts))
        if per_image_t:
            key = key + ("per_image_t",)
        st = self._plans.get(key)
        if st is None:
            if cin != self.conv_in.in_channels:
                raise ValueError(f"input has {cin} channels, conv_in expects {self.conv_in.in_channels}")
            st = self._build_plan(B, h, w, cin, ctx_len, per_image_t)
            if parts is not None:
                self.set_split_inputs(st, parts)
            self._plans[key] = st
            n0 = L.launch_count()
            self._run_plan(st)  # eager warm-up (sets kernel attributes, validates every descriptor)
            st.launches_per_forward = L.launch_count() - n0
            torch.cuda.synchronize()
            if self.use_cuda_graph:
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self._run_plan(st)
                st.graph = g
        return st

    def profile_plan(self, st, iters=3):
        """Per-launch device time of one forward, measured with CUDA events on the launching stream (eager launches
        queued behind a spin kernel, so that host launch time does not leak into the intervals). Returns a list of dicts {op, ms, flops, bytes} in program order; `flops` are algorithmic (2*M*N*K for
        the contraction kernel, 4*B*heads*seq^2*d for attention), `bytes` the minimal operand traffic."""
        stream = torch.cuda.current_stream()
        n = len(st.plan)
        acc = [0.0] * n
        for it in range(iters + 1):
            evs = [torch.cuda.Event(enable_timing=True) for _ in range(n + 1)]
            # The host needs 10 - 20 us per launch through ctypes, most kernels of the small levels less: with an idle
            # GPU the interval between two events is the HOST's time per launch. A spin kernel in front lets the host
            # queue the whole forward first, so the events bracket back-to-back device time as in the graph replay.
            torch.cuda._sleep(int(6e4) * n)
            evs[0].record(stream)
            for i, (fn, a, k) in enumerate(st.plan):
                fn(*a, **k)
                evs[i + 1].record(stream)
            torch.cuda.synchronize()
            if it > 0:
                for i in range(n):
                    acc[i] += evs[i].elapsed_time(evs[i + 1])
        out = []
        for i, (fn, a, k) in enumerate(st.plan):
            rec = {"op": fn.__name__, "ms": acc[i] / iters, "flops": 0, "bytes": 0}
            if fn is ops.gemm:
                a1, w = a[0], a[1]
                M = a1.numel() // a1.shape[-1]
                if k.get("a_stride", 1) == 2:  # the GEMM's rows are the output pixels
                    M = a[2].numel() // a[2].shape[-1]
                # EXECUTED multiply-adds (up2: 4 classes x 4 taps on the low-resolution rows = 4/9 of the 3x3
                # convolution of the up-sampled map it replaces)
                rec["flops"] = 2 * M * w.shape[0] * w.shape[1]
                rec["shape"] = (M, w.shape[0], w.shape[1], k.get("taps", 1))
                rec["bytes"] = 2 * (a1.numel() + (k["a2"].numel() if k.get("a2") is not None else 0) + w.numel()
                                    + M * w.shape[0])
            elif fn is ops.flash_attn:
                rec["flops"] = 4 * k["B"] * k["heads"] * k["seq"] * k["seq"] * k["head_dim"]
                rec["shape"] = (k["B"] * k["heads"], k["seq"], k["head_dim"])
            elif fn is ops.groupnorm:
                x1 = a[0]
                C = a[3].shape[-1]
                rec["bytes"] = 2 * (x1.numel() // x1.shape[-1]) * C * 3  # stats read + apply read + write
            elif fn is ops.layernorm:
                rec["bytes"] = 2 * a[0].numel() * 2
            out.append(rec)
        return out

    def set_split_inputs(self, st, parts):
        """Sampler fast path: read x_t / rgb_latents (/ condition) from separate static buffers so that the channel
        concat of trainers_ldm_cond.py:1134-1141 is fused into conv_in instead of materialised."""
        fn, a, k = st.plan[st.conv_in_slot]
        st.plan[st.conv_in_slot] = (fn, (list(parts),) + a[1:], k)
        st.in_parts = list(parts)

    # ------------------------------------------------------------------ forward (unet.py:281-436)
    @torch.no_grad()
    def forward(self, sample, timestep, encoder_hidden_states=None, class_labels=None, timestep_cond=None,
                attention_mask=None, cross_attention_kwargs=None, down_block_additional_residuals=None,
                mid_block_additional_residual=None, return_dict=True, timestep_img=None):
        if not sample.is_cuda:
            raise L.LdmError("UNet.forward needs CUDA tensors: there is no CPU fallback")
        if self._packed is None:
            self._pack()
        cross, learnable = self._packed["cross"], "object_queries" in self._packed
        if encoder_hidden_states is not None and not cross:
            raise ValueError("encoder_hidden_states given but this UNet has no cross-attention layers "
                             "(remove_cross_attention() was called, tools/main_ldm.py:156-158)")
        if down_block_additional_residuals is not None or mid_block_additional_residual is not None:
            raise NotImplementedError("additional residuals are not on the sampling path")
        B, cin, h, w = sample.shape
        if cin != self.conv_in.in_channels:
            raise ValueError(f"sample has {cin} channels, conv_in expects {self.conv_in.in_channels}")
        use_ehs = cross and not learnable  # unet.py:322-323: learnable object queries replace whatever was passed
        if use_ehs and encoder_hidden_states is None:
            raise ValueError("this UNet keeps its cross-attention layers: encoder_hidden_states is required")
        ts = timestep if torch.is_tensor(timestep) else torch.tensor(timestep)
        # diffusers' convention: a 1-D timestep of B elements gives every image its own timestep
        per_image_t = ts.dim() == 1 and ts.numel() == B and B > 1
        st = self._get_plan(B, h, w, cin, ctx_len=encoder_hidden_states.shape[1] if use_ehs else None,
                            per_image_t=per_image_t)
        if use_ehs:
            self.set_context(st, encoder_hidden_states)
        st.sample.copy_(sample)
        if per_image_t:
            st.timesteps.copy_(ts.to(torch.int64))
        else:
            st.timestep.copy_(ts.reshape(-1)[:1].to(torch.int64))  # unet.py:302-303: one timestep expanded over B
        if st.graph is not None:
            st.graph.replay()
        else:
            self._run_plan(st)
        out = st.out.clone()
        if not return_dict:
            return (out,)
        return UNetOutput(sample=out)

    __call__ = forward
