"""TEST INFRASTRUCTURE - fp32 plain-torch oracle of the first-stage ENCODER and of the img2img sampler steps.

Only tests import this file; the product path (adaprompt_b200/) never does.

A functional, state_dict-driven restatement of ldm/modules/diffusionmodules/model.py (Encoder :408-500, Downsample
:61-79), AutoencoderKL.encode (ldm/models/autoencoder.py:316-320), DiagonalGaussianDistribution
(ldm/modules/distributions/distributions.py:24-44) and DDIMSampler.stochastic_encode / decode (ldm/models/diffusion/
ddim.py:299-350).  It reuses the pinned pieces of oracle/vae_oracle.py (resnet_block, attn_block, the GroupNorm / swish
/ conv helpers, VAESpec) and of oracle/unet_oracle.py (ddim_schedule); Downsample is restated as F.pad followed by the
stride-2 convolution.

Parity unpinned: the reference tree is not available to generate golden encoder outputs, so unlike the decoder oracle
(tests/golden/vae.pt) this restatement is checked against the reference source by reading, not against its outputs.
"""
from __future__ import annotations

from collections import OrderedDict

import numpy as np
import torch
import torch.nn.functional as F

from oracle.unet_oracle import ddim_schedule
from oracle.vae_oracle import SD, VAESpec, _conv, _gn, _swish, attn_block, resnet_block


def encoder_state_spec(spec: VAESpec) -> "OrderedDict[str, tuple]":
    """Key -> shape of encoder.* and quant_conv.*, in the reference's registration order (model.py:436-468,
    autoencoder.py:299)."""
    sp: "OrderedDict[str, tuple]" = OrderedDict()

    def conv(k, co, ci, ks):
        sp[k + ".weight"] = (co, ci, ks, ks)
        sp[k + ".bias"] = (co,)

    def norm(k, c):
        sp[k + ".weight"] = (c,)
        sp[k + ".bias"] = (c,)

    def res(k, ci, co):
        norm(k + ".norm1", ci)
        conv(k + ".conv1", co, ci, 3)
        norm(k + ".norm2", co)
        conv(k + ".conv2", co, co, 3)
        if ci != co:
            conv(k + ".nin_shortcut", co, ci, 1)

    nres = len(spec.ch_mult)
    in_ch_mult = (1,) + spec.ch_mult
    conv("encoder.conv_in", spec.ch, 3, 3)
    block_in = spec.ch
    for i_level in range(nres):
        block_in = spec.ch * in_ch_mult[i_level]
        block_out = spec.ch * spec.ch_mult[i_level]
        for i_block in range(spec.num_res_blocks):
            res(f"encoder.down.{i_level}.block.{i_block}", block_in, block_out)
            block_in = block_out
        if i_level != nres - 1:
            conv(f"encoder.down.{i_level}.downsample.conv", block_in, block_in, 3)
    res("encoder.mid.block_1", block_in, block_in)
    norm("encoder.mid.attn_1.norm", block_in)
    for n in ("q", "k", "v", "proj_out"):
        conv("encoder.mid.attn_1." + n, block_in, block_in, 1)
    res("encoder.mid.block_2", block_in, block_in)
    norm("encoder.norm_out", block_in)
    conv("encoder.conv_out", 2 * spec.z_channels, block_in, 3)
    conv("quant_conv", 2 * spec.embed_dim, 2 * spec.z_channels, 1)
    return sp


def full_state_spec(spec: VAESpec) -> "OrderedDict[str, tuple]":
    """AutoencoderKL with the encoder: encoder.*, decoder.*, quant_conv.*, post_quant_conv.* (autoencoder.py:295-300)."""
    enc = encoder_state_spec(spec)
    dec = spec.state_spec()
    out = OrderedDict((k, v) for k, v in enc.items() if k.startswith("encoder."))
    out.update((k, v) for k, v in dec.items() if k.startswith("decoder."))
    out.update((k, v) for k, v in enc.items() if k.startswith("quant_conv."))
    out.update((k, v) for k, v in dec.items() if k.startswith("post_quant_conv."))
    return out


def downsample(sd: SD, k: str, x: torch.Tensor) -> torch.Tensor:
    """model.py:73-76 (with_conv)."""
    return F.conv2d(F.pad(x, (0, 1, 0, 1), mode="constant", value=0), sd[k + ".weight"], sd[k + ".bias"], stride=2)


def encoder_forward(sd: SD, spec: VAESpec, x: torch.Tensor) -> torch.Tensor:
    """model.py:470-490 (temb None, no attention in the down path)."""
    h = _conv(sd, "encoder.conv_in", x, 1)
    nres = len(spec.ch_mult)
    for i_level in range(nres):
        for i_block in range(spec.num_res_blocks):
            h = resnet_block(sd, f"encoder.down.{i_level}.block.{i_block}", h)
        if i_level != nres - 1:
            h = downsample(sd, f"encoder.down.{i_level}.downsample.conv", h)
    h = resnet_block(sd, "encoder.mid.block_1", h)
    h = attn_block(sd, "encoder.mid.attn_1", h)
    h = resnet_block(sd, "encoder.mid.block_2", h)
    h = _swish(_gn(sd, "encoder.norm_out", h))
    return _conv(sd, "encoder.conv_out", h, 1)


def encode(sd: SD, spec: VAESpec, x: torch.Tensor) -> torch.Tensor:
    """autoencoder.py:316-318: the moments quant_conv(encoder(x))."""
    return _conv(sd, "quant_conv", encoder_forward(sd, spec, x), 0)


def posterior(moments: torch.Tensor):
    """distributions.py:25-33 -> (mean, clamped logvar, std)."""
    mean, logvar = torch.chunk(moments, 2, dim=1)
    logvar = torch.clamp(logvar, -30.0, 20.0)
    return mean, logvar, torch.exp(0.5 * logvar)


def stochastic_encode(x0: torch.Tensor, t_enc: int, S: int, noise: torch.Tensor) -> torch.Tensor:
    """ddim.py:299-312 (DDIM steps, use_original_steps False)."""
    _, alphas, _, _, s1m = ddim_schedule(S)
    a = torch.sqrt(alphas)[t_enc]
    b = torch.as_tensor(np.asarray(s1m)[t_enc], dtype=torch.float32)
    return a * x0 + b * noise


def ddim_decode(apply_model, S: int, x_latent: torch.Tensor, cond, uncond, t_start: int, guidance_scale: float):
    """ddim.py:315-350: t_start DDIM steps from x_latent with eta 0, CFG annealed from guidance_scale towards
    min(2, guidance_scale) by repeated python-float subtraction."""
    ts, alphas, alphas_prev, sigmas, s1m = ddim_schedule(S)
    timesteps = ts[:t_start]
    total = timesteps.shape[0]
    max_g, min_g = guidance_scale, min(2.0, guidance_scale)
    delta = (max_g - min_g) / (total - 1)
    g = max_g
    x = x_latent
    b = x.shape[0]
    for i, step in enumerate(np.flip(timesteps)):
        index = total - i - 1
        t = torch.full((b,), int(step), dtype=torch.long, device=x.device)
        if uncond is None or g == 1.0:
            e_t = apply_model(x, t, cond)
        else:
            c_c, c_in_c, extra = cond
            c_u, c_in_u, _ = uncond
            c2 = (torch.cat([c_c, c_u]), sum([c_in_c, c_in_u], []), extra)
            e_t, e_u = apply_model(torch.cat([x] * 2), torch.cat([t] * 2), c2).chunk(2)
            e_t = e_u + g * (e_t - e_u)
        full = lambda v: torch.full((b, 1, 1, 1), float(v), device=x.device)
        a_t, a_prev, sigma_t, s1m_t = full(alphas[index]), full(alphas_prev[index]), full(sigmas[index]), full(s1m[index])
        pred_x0 = (x - s1m_t * e_t) / a_t.sqrt()
        dir_xt = (1. - a_prev - sigma_t ** 2).sqrt() * e_t
        x = a_prev.sqrt() * pred_x0 + dir_xt
        if i <= total - 1:
            g = g - delta
        else:
            g = 1
    return x


def seeded_images(B: int, H: int, W: int, seed: int) -> torch.Tensor:
    """Seeded images in [-1, 1]: a smooth pattern plus noise, so every layer sees structure at every scale."""
    g = torch.Generator().manual_seed(seed)
    yy, xx = torch.meshgrid(torch.linspace(-1, 1, H), torch.linspace(-1, 1, W), indexing="ij")
    base = torch.stack([torch.sin(3 * xx + 2 * yy), torch.cos(4 * yy - xx), torch.sin(5 * xx * yy)])
    x = 0.7 * base[None] + 0.3 * (torch.rand(B, 3, H, W, generator=g) * 2 - 1)
    return x.clamp(-1, 1)
