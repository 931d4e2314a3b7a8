"""Drop-in front-end with the surface of adaface/adaface_wrapper.py:AdaFaceWrapper :18-296 (reference:
askerlee/adaprompt).

The reference class wraps a `diffusers` StableDiffusionPipeline (its UNet2DConditionModel + DDIMScheduler) and only
uses the reference's own SubjBasisGenerator + CLIP wrappers (SURVEY.md section 3.2).  diffusers / insightface / pretrained
weights are not available offline, so this mirror keeps the constructor and method signatures and drives the
B200-native components instead: adaprompt_b200.clip_text (text encoder with the z_0..z_15 placeholder rows),
adaprompt_b200.subj_basis_generator, adaprompt_b200.unet.UNetModel and adaprompt_b200.ddim.DDIMSampler.  Components are
injected through keyword arguments (`unet`, `text_encoder`, `tokenizer`, `subj_basis_generator`,
`arc2face_text_encoder`, `vae_decoder`, and for pipeline_name="img2img" `vae_encoder`); loading them from `base_model_path` / `adaface_ckpt_path` needs files that
do not exist here and raises a clear error.  End-to-end numerics of the reference wrapper are "parity unpinned"
(diffusers absent, SURVEY.md section 8(c)); its SubjBasisGenerator stage is covered by tests/test_text_gpu.py.
"""
from __future__ import annotations

import re
from typing import Optional

import torch
import torch.nn.functional as F
from torch import nn

from .adaface_util import arc2face_forward_face_embs
from .ddim import DDIMSampler, img2img_t_enc
from .ldm_lite import LatentDiffusionLite

DEFAULT_NEGATIVE_PROMPT = (
    "flaws in the eyes, flaws in the face, lowres, non-HDRi, low quality, worst quality, artifacts, noise, text, "
    "watermark, glitch, mutated, ugly, disfigured, hands, partially rendered objects, partially rendered eyes, "
    "deformed eyeballs, cross-eyed, blurry, mutation, duplicate, out of frame, cropped, mutilated, bad anatomy, "
    "deformed, bad proportions, nude, naked, nsfw, topless, bare breasts")


class AdaFaceWrapper(nn.Module):
    def __init__(self, pipeline_name, base_model_path, adaface_ckpt_path, device, subject_string="z", num_vectors=16,
                 num_inference_steps=50, negative_prompt=None, use_840k_vae=False, use_ds_text_encoder=False,
                 is_training=False, *, unet=None, text_encoder=None, tokenizer=None, subj_basis_generator=None,
                 arc2face_text_encoder=None, vae_decoder=None, vae_encoder=None):
        super().__init__()
        self.pipeline_name = pipeline_name
        self.base_model_path = base_model_path
        self.adaface_ckpt_path = adaface_ckpt_path
        self.use_840k_vae = use_840k_vae
        self.use_ds_text_encoder = use_ds_text_encoder
        self.subject_string = subject_string
        self.num_vectors = num_vectors
        self.num_inference_steps = num_inference_steps
        self.device = device
        self.is_training = is_training
        self._injected = dict(unet=unet, text_encoder=text_encoder, tokenizer=tokenizer,
                              subj_basis_generator=subj_basis_generator, arc2face_text_encoder=arc2face_text_encoder,
                              vae_decoder=vae_decoder, vae_encoder=vae_encoder)
        self.initialize_pipeline()
        self.extend_tokenizer_and_text_encoder()
        self.negative_prompt = DEFAULT_NEGATIVE_PROMPT if negative_prompt is None else negative_prompt

    # ------------------------------------------------------------------ loading (adaface_wrapper.py:49-150)
    def load_subj_basis_generator(self, adaface_ckpt_path):
        sbg = self._injected["subj_basis_generator"]
        if sbg is None:
            # Reference checkpoints are pickled nn.Module objects (embedding_manager.py:1824-1838); checkpoint.py unpickles
            # them without the reference package and converts to the native SubjBasisGenerator (adaface_wrapper.py:50-57).
            from .checkpoint import load_adaface_ckpt
            ckpt = load_adaface_ckpt(adaface_ckpt_path, clip_tokenizer=self._injected["tokenizer"])
            sbgs = ckpt["string_to_subj_basis_generator_dict"]
            if self.subject_string not in sbgs:
                raise KeyError(f"Subject '{self.subject_string}' not found in the embedding manager checkpoint "
                               f"(has {sorted(sbgs)})")
            sbg = sbgs[self.subject_string]
        self.subj_basis_generator = sbg
        self.subj_basis_generator.num_out_layers = 1                                                 # :59
        self.subj_basis_generator.to(self.device)
        self.subj_basis_generator.train(self.is_training)

    def initialize_pipeline(self):
        self.load_subj_basis_generator(self.adaface_ckpt_path)
        inj = self._injected
        if inj["arc2face_text_encoder"] is None or inj["text_encoder"] is None or inj["tokenizer"] is None:
            raise FileNotFoundError("text_encoder / tokenizer / arc2face_text_encoder must be injected: pretrained "
                                    f"weights under {self.base_model_path!r} and 'models/arc2face' are not available offline")
        self.arc2face_text_encoder = inj["arc2face_text_encoder"].to(self.device)
        self.text_encoder = inj["text_encoder"].to(self.device)      # clip_text.CLIPTextModelWrapper
        self.tokenizer = inj["tokenizer"]
        self.vae_decoder = inj["vae_decoder"]
        self.vae_encoder = inj["vae_encoder"]          # vae.AutoencoderKL(with_encoder=True): img2img from RGB images
        if self.pipeline_name is not None:
            if inj["unet"] is None:
                raise FileNotFoundError("unet must be injected (adaprompt_b200.unet.UNetModel with SD-1.5 weights)")
            self.ldm = LatentDiffusionLite(inj["unet"]).to(self.device)
            self.sampler = DDIMSampler(self.ldm)
        else:
            self.ldm = self.sampler = None                                                           # :141-146: no unet / vae
        if getattr(self.subj_basis_generator, "clip_tokenizer", None) is None:                       # :148-150
            self.subj_basis_generator.clip_tokenizer = self.tokenizer

    def extend_tokenizer_and_text_encoder(self):
        """:152-182: add z_0 .. z_{n-1} to the tokenizer and grow the token-embedding table."""
        if self.num_vectors < 1:
            raise ValueError(f"num_vectors has to be larger or equal to 1, but is {self.num_vectors}")
        self.placeholder_tokens = [f"{self.subject_string}_{i}" for i in range(self.num_vectors)]
        self.placeholder_tokens_str = " ".join(self.placeholder_tokens)
        emb = self.text_encoder.text_model.embeddings.token_embedding
        old_n = emb.weight.shape[0]
        if hasattr(self.tokenizer, "add_tokens"):
            added = self.tokenizer.add_tokens(self.placeholder_tokens)
            if added != self.num_vectors:
                raise ValueError(f"The tokenizer already contains the token {self.subject_string}. Please pass a "
                                 "different `subject_string` that is not already in the tokenizer.")
            self.placeholder_token_ids = self.tokenizer.convert_tokens_to_ids(self.placeholder_tokens)
        else:
            self.placeholder_token_ids = list(range(old_n, old_n + self.num_vectors))
        new = nn.Embedding(old_n + self.num_vectors, emb.weight.shape[1]).to(emb.weight.device)
        with torch.no_grad():
            new.weight[:old_n] = emb.weight
            new.weight[old_n:] = emb.weight[:old_n].mean(0, keepdim=True)
        self.text_encoder.text_model.embeddings.token_embedding = new

    def update_text_encoder_subj_embs(self, subj_embs):
        """:184-190: subj_embs [16, 768] -> rows of the token-embedding table."""
        token_embeds = self.text_encoder.text_model.embeddings.token_embedding.weight.data
        with torch.no_grad():
            for i, token_id in enumerate(self.placeholder_token_ids):
                token_embeds[token_id] = subj_embs[i]

    def update_prompt(self, prompt):
        """:192-204."""
        if self.placeholder_tokens_str in prompt:
            return prompt
        if re.search(r"\b" + self.subject_string + r"\b", prompt) is None:
            return self.placeholder_tokens_str + " " + prompt
        return re.sub(r"\b" + self.subject_string + r"\b", self.placeholder_tokens_str, prompt)

    # ------------------------------------------------------------------ embeddings (:207-254)
    def generate_adaface_embeddings(self, image_paths, image_folder=None, pre_face_embs=None, gen_rand_face=False,
                                    out_id_embs_scale=1., noise_level=0, update_text_encoder=True):
        if pre_face_embs is not None:
            faceid_embeds = pre_face_embs.to(self.device).float()
        elif gen_rand_face:
            faceid_embeds = torch.randn(1, 512, device=self.device)
        else:
            raise NotImplementedError("face detection / ArcFace feature extraction (insightface) is out of scope; pass "
                                      "pre_face_embs or gen_rand_face=True")
        if noise_level > 0:                                                                          # adaface/util.py:300-307
            faceid_embeds = faceid_embeds + torch.randn_like(faceid_embeds) * faceid_embeds.std() * noise_level
        faceid_embeds = F.normalize(faceid_embeds, p=2, dim=-1)                                      # adaface/util.py:311
        with torch.no_grad():
            id_prompt_emb = arc2face_forward_face_embs(self.tokenizer, self.arc2face_text_encoder, faceid_embeds,
                                                       input_max_length=22, return_full_and_core_embs=False)  # :234
            adaface_subj_embs, _ = self.subj_basis_generator(id_prompt_emb, None, None, out_id_embs_scale=out_id_embs_scale,
                                                             is_face=True, is_training=False,
                                                             adaface_prompt_embs_inf_type="full_half_pad")    # :246
        adaface_subj_embs = adaface_subj_embs.squeeze()                                              # [1,1,16,768] -> [16,768]
        if update_text_encoder:
            self.update_text_encoder_subj_embs(adaface_subj_embs)
        return adaface_subj_embs

    def _tokenize(self, text):
        enc = self.tokenizer(text, truncation=True, padding="max_length", max_length=77, return_tensors="pt")
        return (enc["input_ids"] if isinstance(enc, dict) else enc.input_ids).to(self.device)

    def encode_prompt(self, prompt, negative_prompt=None, device="cuda", verbose=False):
        """:256-271 -> (prompt_embeds [1,77,768], negative_prompt_embeds [1,77,768])."""
        if negative_prompt is None:
            negative_prompt = self.negative_prompt
        prompt = self.update_prompt(prompt)
        if verbose:
            print(f"Prompt: {prompt}")
        with torch.no_grad():
            pe = self.text_encoder(input_ids=self._tokenize(prompt))[0]
            ne = self.text_encoder(input_ids=self._tokenize(negative_prompt))[0]
        return pe, ne

    # ------------------------------------------------------------------ sampling (:274-296)
    def forward(self, noise, prompt, negative_prompt=None, guidance_scale=4.0, out_image_count=4, ref_img_strength=0.8,
                generator=None, verbose=False):
        if self.sampler is None:
            raise RuntimeError("pipeline_name=None: the wrapper was built without a UNet")
        t_enc = None
        if self.pipeline_name == "img2img":
            # host-side checks before any device work (a t_enc out of range would fault inside stochastic_encode)
            t_enc = img2img_t_enc(ref_img_strength, self.num_inference_steps)
            if noise.dim() != 4 or noise.shape[1] not in (3, 4):
                raise ValueError("img2img: `noise` must be an NCHW image in [-1, 1] (3 channels) or latents (4 channels)")
            if noise.shape[1] == 3 and self.vae_encoder is None:
                raise RuntimeError("img2img from an RGB image needs vae_encoder (vae.AutoencoderKL(with_encoder=True))")
        pe, ne = self.encode_prompt(prompt, negative_prompt, device=self.device, verbose=verbose)
        b = out_image_count
        # the LDM UNet takes one context per cross-attention layer: the same prompt embedding for all 16
        c = pe.repeat(b * 16, 1, 1).contiguous()
        uc = ne.repeat(b * 16, 1, 1).contiguous()
        extra = {"use_layerwise_context": True, "use_conv_attn_kernel_size": -1, "placeholder2indices": None,
                 "is_training": False}
        noise = noise.to(self.device).float()
        g = float(guidance_scale)
        if t_enc is not None:
            samples = self._img2img(noise, b, c, uc, [prompt] * b, [negative_prompt or self.negative_prompt] * b, extra, g,
                                    t_enc)
        else:
            samples, _ = self.sampler.sample(self.num_inference_steps, b, list(noise.shape[1:]),
                                             conditioning=(c, [prompt] * b, dict(extra)),
                                             unconditional_conditioning=(uc, [negative_prompt or self.negative_prompt] * b,
                                                                         dict(extra)),
                                             guidance_scale=(g, g), eta=0.0, x_T=noise, verbose=False)
        if self.vae_decoder is None:
            return samples          # latents; the VAE decoder is SURVEY.md section 8(f) row N1 ("next")
        return self.vae_decoder(samples / self.ldm.scale_factor)

    def _img2img(self, init, b, c, uc, prompts, neg_prompts, extra, g, t_enc):
        """SD scripts/img2img.py on the LDM sampler: encode (3-channel images; 4 channels are latents already, as in
        diffusers' img2img pipeline), stochastic_encode to step t_enc, then DDIMSampler.decode with CFG."""
        if init.shape[1] == 3:
            from .vae import encode_first_stage
            init = self.ldm.get_first_stage_encoding(encode_first_stage(self.vae_encoder, init))
        if init.shape[0] != b:
            if init.shape[0] != 1:
                raise ValueError(f"img2img: {init.shape[0]} init images for out_image_count {b}")
            init = init.repeat(b, 1, 1, 1)
        self.sampler.make_schedule(ddim_num_steps=self.num_inference_steps, ddim_eta=0.0, verbose=False)
        z_enc = self.sampler.stochastic_encode(init, torch.full((b,), t_enc, dtype=torch.long, device=init.device))
        return self.sampler.decode(z_enc, (c, prompts, dict(extra)), t_enc, guidance_scale=g,
                                   unconditional_conditioning=(uc, neg_prompts, dict(extra)))
