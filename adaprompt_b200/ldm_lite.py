"""Adapter slice of ldm/models/diffusion/ddpm.py that sits between the sampler and the UNet:
register_schedule :240-292, q_sample :416-419, apply_model :2192-2297 (live line :2292) and
DiffusionWrapper.forward :5514-5544 (crossattn branch).  Everything else in ddpm.py (the Lightning
training module, losses, optimisers) is out of scope (SURVEY.md section 8)."""
from __future__ import annotations

from functools import partial

import numpy as np
import torch
from torch import nn

from .diffusion_util import make_beta_schedule
from .unet import UNetModel

SD15_UNET_CONFIG = dict(  # configs/stable-diffusion/v1-inference-ada.yaml:35-51
    image_size=32, in_channels=4, out_channels=4, model_channels=320, attention_resolutions=[4, 2, 1],
    num_res_blocks=2, channel_mult=[1, 2, 4, 4], num_heads=8, use_spatial_transformer=True,
    transformer_depth=1, context_dim=768, use_checkpoint=True, legacy=False)


class DiffusionWrapper(nn.Module):
    """ddpm.py:5505-5544: unpacks the (c_static_emb, c_in, extra_info) conditioning tuple."""

    def __init__(self, diffusion_model: nn.Module, conditioning_key="crossattn"):
        super().__init__()
        self.diffusion_model = diffusion_model
        self.conditioning_key = conditioning_key
        assert conditioning_key == "crossattn", "only the crossattn branch is used by AdaFace"

    def forward(self, x, t, c_concat=None, c_crossattn=None):
        c_static_emb, c_in, extra_info = c_crossattn[0]                         # :5522-5524
        return self.diffusion_model(x, t, context=c_static_emb, context_in=c_in, extra_info=extra_info)  # :5533


class LatentDiffusionLite(nn.Module):
    """What DDIMSampler needs from LatentDiffusion: betas / alphas_cumprod(_prev) / num_timesteps / device /
    apply_model / q_sample, with the SD-1.5 'linear' schedule (v1-inference-ada.yaml:5-9)."""

    def __init__(self, unet: nn.Module = None, timesteps=1000, linear_start=0.00085, linear_end=0.012,
                 beta_schedule="linear", scale_factor=0.18215, parameterization="eps", cond_stage_model=None,
                 embedding_manager=None, first_stage_model=None):
        super().__init__()
        self.model = DiffusionWrapper(unet if unet is not None else UNetModel(**SD15_UNET_CONFIG))
        self.cond_stage_model = cond_stage_model      # clip_text.FrozenCLIPEmbedder (ddpm.py:756)
        self.embedding_manager = embedding_manager    # embedding_manager.EmbeddingManagerLite (ddpm.py:793)
        self.first_stage_model = first_stage_model    # vae.AutoencoderKL (ddpm.py:744-751); encodes if built with_encoder
        self.use_layerwise_embedding = True           # v1-inference-ada.yaml:19
        self.N_CA_LAYERS = 16                         # ddpm.py:150
        self.empty_context = None
        self.compel_cfg_weight_level_range = None
        self.apply_compel_cfg_prob = 0
        self.parameterization = parameterization
        self.scale_factor = scale_factor
        self.register_schedule(beta_schedule, timesteps, linear_start, linear_end)

    def register_schedule(self, beta_schedule, timesteps, linear_start, linear_end, cosine_s=8e-3):
        """ddpm.py:240-292 (the buffers the sampling path reads)."""
        betas = make_beta_schedule(beta_schedule, timesteps, linear_start=linear_start, linear_end=linear_end,
                                   cosine_s=cosine_s)
        alphas = 1. - betas
        alphas_cumprod = np.cumprod(alphas, axis=0)
        alphas_cumprod_prev = np.append(1., alphas_cumprod[:-1])
        self.num_timesteps = int(betas.shape[0])
        to_torch = partial(torch.tensor, dtype=torch.float32)
        self.register_buffer("betas", to_torch(betas))
        self.register_buffer("alphas_cumprod", to_torch(alphas_cumprod))
        self.register_buffer("alphas_cumprod_prev", to_torch(alphas_cumprod_prev))
        self.register_buffer("sqrt_alphas_cumprod", to_torch(np.sqrt(alphas_cumprod)))
        self.register_buffer("sqrt_one_minus_alphas_cumprod", to_torch(np.sqrt(1. - alphas_cumprod)))

    @property
    def device(self):
        return self.betas.device

    def q_sample(self, x_start, t, noise=None):
        """ddpm.py:416-419."""
        noise = torch.randn_like(x_start) if noise is None else noise
        a = self.sqrt_alphas_cumprod[t].reshape(-1, *((1,) * (x_start.dim() - 1)))
        b = self.sqrt_one_minus_alphas_cumprod[t].reshape(-1, *((1,) * (x_start.dim() - 1)))
        return a * x_start + b * noise

    def get_learned_conditioning(self, cond_in, zs_clip_features=None, zs_id_embs=None,
                                 zs_out_id_embs_scale_range=(1.0, 1.0), randomize_clip_weights=False,
                                 apply_arc2face_inverse_embs=False, apply_arc2face_embs=False, embman_iter_type=None):
        """ddpm.py:970-1085, inference path: prompts (or token ids) -> (static_prompt_embedding [16*B, 77, 768],
        cond_in, extra_info).  The uncond prompt passes no zs features and so reuses none."""
        if randomize_clip_weights or apply_arc2face_inverse_embs or apply_arc2face_embs:
            raise NotImplementedError("training / Arc2Face-evaluation conditioning variants")
        if self.cond_stage_model is None or self.embedding_manager is None:
            raise RuntimeError("LatentDiffusionLite: cond_stage_model / embedding_manager are not set")
        if zs_clip_features is not None or zs_id_embs is not None:
            self.embedding_manager.set_zs_image_features(zs_clip_features, zs_id_embs,
                                                         zs_out_id_embs_scale_range=zs_out_id_embs_scale_range)
            apply_compel_cfg_prob = 0                                                               # :994
        else:
            apply_compel_cfg_prob = self.apply_compel_cfg_prob
        self.embedding_manager.iter_type = embman_iter_type or "recon_iter"                         # :1008
        static_prompt_embedding = self.cond_stage_model.encode(cond_in, embedding_manager=self.embedding_manager)  # :1011
        import copy
        extra_info = {                                                                              # :1065-1076
            "use_layerwise_context": self.use_layerwise_embedding,
            "use_conv_attn_kernel_size": getattr(self.embedding_manager, "use_conv_attn_kernel_size", -1),
            "placeholder2indices": copy.copy(self.embedding_manager.placeholder2indices),
            "prompt_emb_mask": copy.copy(self.embedding_manager.prompt_emb_mask),
            "is_training": self.embedding_manager.training,
            "compel_cfg_weight_level_range": self.compel_cfg_weight_level_range,
            "apply_compel_cfg_prob": apply_compel_cfg_prob,
            "empty_context": self.empty_context,
            "capture_distill_attn": False,
        }
        return (static_prompt_embedding, cond_in, extra_info)                                       # :1078

    @torch.no_grad()
    def decode_first_stage(self, z, predict_cids=False, force_not_quantize=False, max_batch=None):
        """ddpm.py:1260-1318, the plain branch (no VQ codebook, no split_input_params): latents -> RGB in [-1, 1]."""
        if predict_cids or hasattr(self, "split_input_params"):
            raise NotImplementedError("decode_first_stage: VQ / patch-split decoding is not used by AdaFace sampling")
        if self.first_stage_model is None:
            raise RuntimeError("LatentDiffusionLite: first_stage_model is not set")
        from .vae import decode_first_stage
        return decode_first_stage(self.first_stage_model, z, self.scale_factor, max_batch=max_batch)

    @torch.no_grad()
    def encode_first_stage(self, x, max_batch=None):
        """ddpm.py encode_first_stage, the plain branch (no split_input_params): NCHW images in [-1, 1] -> the posterior
        (needs first_stage_model built with_encoder=True)."""
        if hasattr(self, "split_input_params"):
            raise NotImplementedError("encode_first_stage: patch-split encoding is not used by AdaFace sampling")
        if self.first_stage_model is None:
            raise RuntimeError("LatentDiffusionLite: first_stage_model is not set")
        from .vae import encode_first_stage
        return encode_first_stage(self.first_stage_model, x, max_batch=max_batch)

    def get_first_stage_encoding(self, encoder_posterior):
        """ddpm.py get_first_stage_encoding: scale_factor * posterior.sample() (one fused kernel), or scale_factor * a
        tensor."""
        from .vae import DiagonalGaussianDistribution
        if isinstance(encoder_posterior, DiagonalGaussianDistribution):
            return encoder_posterior.scaled_sample(self.scale_factor)
        if isinstance(encoder_posterior, torch.Tensor):
            return self.scale_factor * encoder_posterior
        raise NotImplementedError(f"encoder_posterior of type '{type(encoder_posterior)}' not yet implemented")

    def refresh_conditioning(self, cond, batch: int):
        """Hook for the CUDA-graph sampler: (re)project the conditioning tuple's context through the 16
        cross-attention to_k / to_v layers now - in place when `cond[0]` is a static buffer whose content
        changed.  Returns the {layer: ContextKV} dict so the caller can detect re-allocation."""
        c_static_emb, _, extra_info = cond
        iter_type = (extra_info or {}).get("iter_type", "normal_recon")
        return self.model.diffusion_model.context_kv(c_static_emb, batch, iter_type)

    def time_embedding_rows(self, timesteps: torch.Tensor):
        """Hook for the CUDA-graph sampler: every ResBlock's emb_layers(time_embed(t)) for a vector of timesteps, [len(t),
        sum Cout] - the part of the UNet forward that depends on t alone, hoisted out of the 50-step loop (the sampler
        hands the row of the current step back through extra_info['emb_rows'])."""
        return self.model.diffusion_model.time_embedding(timesteps)[1]

    def apply_model(self, x_noisy, t, cond, return_ids=False):
        """ddpm.py:2192-2201,2292."""
        if not isinstance(cond, dict):
            if not isinstance(cond, list):
                cond = [cond]
            cond = {"c_crossattn": cond}
        return self.model(x_noisy, t, **cond)
