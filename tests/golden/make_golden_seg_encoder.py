"""Golden fixture for the seg-AE ENCODER side (SURVEY.md section 8f rank 3): runs the REAL reference
``GeneralVAESeg`` (ldmseg/models/vae.py:175-307; encoder, DiagonalGaussianDistribution, forward) on a seeded input and
stores its state_dict, the moments, the posterior's mode / std and ``forward(sample_posterior=False)``.
Authoring container only (needs /root/reference).

    python tests/golden/make_golden_seg_encoder.py     -> tests/golden/seg_encoder_small.npz
                                                          tests/golden/seg_encoder_small_part2.npz

Random float32 weights do not compress, so the arrays are spread over two files to keep each under 1 MB: the input,
the outputs, cfg and the encoder's output convolution go to the second one.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import ref_stubs  # noqa: E402

ref_stubs.install()
from ldmseg.models.vae import GeneralVAESeg  # noqa: E402

CFG = dict(in_channels=16, int_channels=64, out_channels=16, block_out_channels=(16, 32, 64, 128), latent_channels=4,
           num_latents=2, num_upscalers=2, upscale_channels=64, norm_num_groups=32, scaling_factor=0.2,
           parametrization="gaussian", act_fn="none", num_mid_blocks=0)


def main():
    torch.manual_seed(5)
    vae = GeneralVAESeg(**CFG).eval()
    g = torch.Generator().manual_seed(6)
    with torch.no_grad():
        for p in vae.parameters():  # non-trivial biases / norm affine parameters
            if p.dim() == 1:
                p.add_(0.1 * torch.randn(p.shape, generator=g))
    bits = (torch.rand((2, 16, 32, 48), generator=g) < 0.5).float() * 2 - 1
    bits[:, :, :3, :5] = 0.5  # an "ignore" patch (encode_bitmap fill_value)
    with torch.no_grad():
        post = vae.encode(bits).latent_dist
        out = vae(bits, sample_posterior=False)
    sd = {k: v.numpy() for k, v in vae.state_dict().items()}
    arrays = dict(bits=bits.numpy(), moments=post.parameters.numpy(), mode=post.mode().numpy(), std=post.std.numpy(),
                  forward=out.sample.numpy(), cfg=np.array(repr(CFG)), **{"sd." + k: v for k, v in sd.items()})
    part2 = {"bits", "moments", "mode", "std", "forward", "cfg", "sd.encoder.15.weight", "sd.encoder.15.bias"}
    np.savez_compressed(os.path.join(HERE, "seg_encoder_small.npz"), **{k: v for k, v in arrays.items() if k not in part2})
    np.savez_compressed(os.path.join(HERE, "seg_encoder_small_part2.npz"), **{k: v for k, v in arrays.items() if k in part2})
    print("wrote seg_encoder_small.npz", post.parameters.shape, out.sample.shape, sorted(k for k in sd if k.startswith("encoder"))[:12])


if __name__ == "__main__":
    main()
