"""CPU restatement (plain torch fp32) of the reference VAE decode - TEST INFRASTRUCTURE for the SURVEY 8(f) rank-1
"next" row; nothing on the product path imports it.

    AutoencoderKL.decode      ldm/models/autoencoder.py:40-44       z / scale_factor -> post_quant_conv -> Decoder
    Decoder.forward           ldm/modules/diffusionmodules/model.py:535-568
    ResnetBlock.forward       model.py:121-141   (temb is None in the VAE: temb_ch = 0)
    AttnBlock.forward         model.py:178-202   (single head over H*W tokens, scale C^-0.5)
    Upsample.forward          model.py:53-57     (nearest x2, then 3x3 conv)
    Normalize                 model.py:38-39     (GroupNorm 32 groups, eps 1e-6)

    AutoencoderKL.encode      autoencoder.py:34-38   Encoder -> quant_conv -> DiagonalGaussianDistribution.sample() * scale_factor
    Encoder.forward           model.py:434-459
    Downsample.forward        model.py:73-77         (F.pad (0,1,0,1), then 3x3 stride-2 conv without padding)
    DiagonalGaussianDistribution  ldm/modules/distributions/distributions.py:24-37 (logvar clamped to [-30, 20]; the noise is
                              drawn on the CPU with the global generator and moved to the device)

Pinned by oracle/gen_golden.py --vae: executed against the unmodified reference AutoencoderKL with the same synthetic
weights (measured difference recorded in tests/golden/*_vae_*.pt["oracle_max_abs_diff"]).
"""
from __future__ import annotations

from typing import Dict

import torch
import torch.nn.functional as F


def _gn(x, sd, prefix):
    return F.group_norm(x, 32, sd[prefix + ".weight"], sd[prefix + ".bias"], eps=1e-6)


def _conv(x, sd, prefix, pad):
    return F.conv2d(x, sd[prefix + ".weight"], sd[prefix + ".bias"], padding=pad)


def _swish(x):
    return x * torch.sigmoid(x)


def resnet_block(x, sd, prefix):
    h = _conv(_swish(_gn(x, sd, prefix + ".norm1")), sd, prefix + ".conv1", 1)
    h = _conv(_swish(_gn(h, sd, prefix + ".norm2")), sd, prefix + ".conv2", 1)       # dropout = 0 in eval
    if prefix + ".nin_shortcut.weight" in sd:
        x = _conv(x, sd, prefix + ".nin_shortcut", 0)
    return x + h


def attn_block(x, sd, prefix):
    h = _gn(x, sd, prefix + ".norm")
    q, k, v = (_conv(h, sd, f"{prefix}.{n}", 0) for n in ("q", "k", "v"))
    b, c, hh, ww = q.shape
    q = q.reshape(b, c, hh * ww).permute(0, 2, 1)                     # b, hw, c
    k = k.reshape(b, c, hh * ww)                                      # b, c, hw
    w = torch.softmax(torch.bmm(q, k) * (int(c) ** -0.5), dim=2)      # b, hw(q), hw(k)
    v = v.reshape(b, c, hh * ww)
    h = torch.bmm(v, w.permute(0, 2, 1)).reshape(b, c, hh, ww)        # h[b,c,j] = sum_i v[b,c,i] w[b,j,i]
    return x + _conv(h, sd, prefix + ".proj_out", 0)


@torch.no_grad()
def encode_test_image(cfg, B: int, seed: int) -> torch.Tensor:
    """The encoder fixtures' input: a smooth image in [-1, 1] plus seeded texture (what `encode` sees: a normalised RGB
    picture).  Fixtures too large to store it keep its sha256 instead (oracle/gen_golden.py run_vae_encode)."""
    g = torch.Generator().manual_seed(seed)
    S = cfg.image_size
    yy, xx = torch.meshgrid(torch.linspace(-1, 1, S), torch.linspace(-1, 1, S), indexing="ij")
    base = torch.stack([torch.sin(3 * xx + c) * torch.cos(2 * yy - c) for c in range(cfg.in_channels)], 0)
    return (0.7 * base[None] + 0.3 * torch.randn(B, cfg.in_channels, S, S, generator=g)).clamp(-1, 1)


def vae_decode(cfg, sd: Dict[str, torch.Tensor], z: torch.Tensor) -> torch.Tensor:
    """z: [B, embed_dim, h, w] (the sampler's latent) -> image [B, out_ch, h * 2^(levels-1), w * 2^(levels-1)]."""
    z = (1.0 / cfg.scale_factor) * z
    h = _conv(z, sd, "post_quant_conv", 0)
    h = _conv(h, sd, "decoder.conv_in", 1)
    h = resnet_block(h, sd, "decoder.mid.block_1")
    h = attn_block(h, sd, "decoder.mid.attn_1")
    h = resnet_block(h, sd, "decoder.mid.block_2")
    for i_level in reversed(range(len(cfg.ch_mult))):
        for i_block in range(cfg.num_res_blocks + 1):
            h = resnet_block(h, sd, f"decoder.up.{i_level}.block.{i_block}")
        if i_level != 0:
            h = F.interpolate(h, scale_factor=2.0, mode="nearest")
            h = _conv(h, sd, f"decoder.up.{i_level}.upsample.conv", 1)
    h = _swish(_gn(h, sd, "decoder.norm_out"))
    return _conv(h, sd, "decoder.conv_out", 1)


@torch.no_grad()
def vae_encode_moments(cfg, sd: Dict[str, torch.Tensor], x: torch.Tensor) -> torch.Tensor:
    """x: image [B, in_channels, H, W] in [-1, 1] -> moments [B, 2 * embed_dim, H / 2^(levels-1), ...] (mean | logvar)."""
    h = _conv(x, sd, "encoder.conv_in", 1)
    nlev = len(cfg.ch_mult)
    for i_level in range(nlev):
        for i_block in range(cfg.num_res_blocks):
            h = resnet_block(h, sd, f"encoder.down.{i_level}.block.{i_block}")
        if i_level != nlev - 1:
            p = f"encoder.down.{i_level}.downsample.conv"
            h = F.conv2d(F.pad(h, (0, 1, 0, 1)), sd[p + ".weight"], sd[p + ".bias"], stride=2)
    h = resnet_block(h, sd, "encoder.mid.block_1")
    h = attn_block(h, sd, "encoder.mid.attn_1")
    h = resnet_block(h, sd, "encoder.mid.block_2")
    h = _conv(_swish(_gn(h, sd, "encoder.norm_out")), sd, "encoder.conv_out", 1)
    return _conv(h, sd, "quant_conv", 0)


@torch.no_grad()
def vae_encode(cfg, sd: Dict[str, torch.Tensor], x: torch.Tensor) -> torch.Tensor:
    """encode(x): one posterior sample times scale_factor; consumes torch's global CPU generator like the reference."""
    mean, logvar = torch.chunk(vae_encode_moments(cfg, sd, x), 2, dim=1)
    std = torch.exp(0.5 * torch.clamp(logvar, -30.0, 20.0))
    return (mean + std * torch.randn(mean.shape).to(x.device)) * cfg.scale_factor
