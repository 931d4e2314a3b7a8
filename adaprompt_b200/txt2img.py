"""Command-line sampler with the core options of scripts/stable_txt2img.py (reference: askerlee/adaprompt :37-300 argument
parser, :324-687 main) on the B200 components - SURVEY.md section 8(f) row N3.

    python -m adaprompt_b200.txt2img --prompt "a photo of a z" --scale 4 1 --n_samples 8 --bs 8 --ddim_steps 50 \\
        --ckpt models/stable-diffusion-v-1-5/v1-5-dste8-vae.ckpt --tokenizer_dir models/clip-vit-large-patch14 \\
        --subj_ckpt adaface_sbg_state_dict.pt --face_embs id_embs.pt --outdir outputs
    torchrun --nproc-per-node 8 -m adaprompt_b200.txt2img ...        # images sharded over the GPUs, no collective

Pipeline (same order as stable_txt2img.py:560-687): face ID embeddings -> EmbeddingManager.set_zs_image_features ->
get_learned_conditioning(prompts) and (negative prompts) -> DDIMSampler.sample with the annealed (max, min) guidance
pair -> decode_first_stage -> clamp((x + 1) / 2) -> PNG files and a grid.

What the reference CLI does that this one does not: face detection / ArcFace feature extraction from `--ref_images`
(insightface; pass pre-computed 512-d embeddings with --face_embs instead), CLIP / face-similarity scoring
(--scores_csv, --calc_face_sim, --compare_with), DreamBooth / class-prompt comparison modes, and un-pickling the
reference's nn.Module checkpoints (embedding_manager.py:1824-1838 stores module OBJECTS; --subj_ckpt takes a plain
state_dict of SubjBasisGenerator).  `--synthetic` runs the whole pipeline on random-init weights of the real
architecture with a hashing stand-in tokenizer (no vocabulary or checkpoint files exist offline): that is what the
GPU test drives end to end.

img2img (SD scripts/img2img.py): with --init_img the image (--W x --H pixels) is encoded by the VAE encoder, its latent
is noised to step t_enc = int(--strength * --ddim_steps) by DDIMSampler.stochastic_encode and denoised by
DDIMSampler.decode, whose guidance scale anneals from the first --scale value towards min(2, scale).
"""
from __future__ import annotations

import argparse
import os
import sys
import types
import zlib
from typing import Dict, List, Optional

import torch

BOS, EOS = 49406, 49407
TOK_COMMA, TOK_Z, TOK_Y = 267, 345, 344          # ldm/modules/embedding_manager.py:1062


class HashTokenizer:
    """Stand-in with the CLIPTokenizer call protocol for --synthetic runs: whitespace / comma split, the subject and
    background strings and ',' keep their real CLIP ids, every other word hashes into the vocabulary."""
    pad_token_id = EOS

    def __init__(self, fixed: Optional[Dict[str, int]] = None):
        self.fixed = {",": TOK_COMMA, "z": TOK_Z, "y": TOK_Y, "photo": 1125, "of": 539, "a": 320, "id": 1014,
                      "person": 2533}
        self.fixed.update(fixed or {})

    def _ids(self, text: str) -> List[int]:
        return [self.fixed.get(w, 1000 + zlib.crc32(w.encode()) % 40000) for w in text.lower().replace(",", " , ").split()]

    def encode(self, text, add_special_tokens=False):
        return self._ids(text)

    def __call__(self, text, truncation=True, padding="max_length", max_length=77, return_tensors="pt", **kw):
        texts = [text] if isinstance(text, str) else list(text)
        rows = []
        for t in texts:
            ids = [BOS] + self._ids(t)[:max_length - 2] + [EOS]
            rows.append(ids + [EOS] * (max_length - len(ids)))
        return types.SimpleNamespace(input_ids=torch.tensor(rows, dtype=torch.long))


def split_sd15_checkpoint(sd: Dict[str, torch.Tensor]) -> Dict[str, Dict[str, torch.Tensor]]:
    """An SD-1.5 / AdaFace LatentDiffusion checkpoint (`state_dict` of ddpm.py:LatentDiffusion) -> per-component
    state_dicts with the prefixes stripped: model.diffusion_model.* (UNetModel), first_stage_model.* (AutoencoderKL),
    cond_stage_model.transformer.* (the HF CLIPTextModel inside FrozenCLIPEmbedder, modules.py:195)."""
    sd = sd.get("state_dict", sd)
    out = {"unet": {}, "vae": {}, "clip": {}}
    for k, v in sd.items():
        for prefix, name in (("model.diffusion_model.", "unet"), ("first_stage_model.", "vae"),
                             ("cond_stage_model.transformer.", "clip")):
            if k.startswith(prefix):
                out[name][k[len(prefix):]] = v
    return out


def build_pipeline(args, device):
    """Instantiates UNet / VAE / FrozenCLIPEmbedder / EmbeddingManager / SubjBasisGenerator on `device` and loads
    either the checkpoint files or the synthetic-weight recipe."""
    from .clip_text import CLIPTextConfigLite, CLIPTextModelWrapper, FrozenCLIPEmbedder
    from .embedding_manager import EmbeddingManagerLite
    from .ldm_lite import SD15_UNET_CONFIG, LatentDiffusionLite
    from .subj_basis_generator import SubjBasisGenerator
    from .unet import UNetModel
    from .vae import AutoencoderKL
    from .weights import spec_of, synth_state_dict

    if args.synthetic:
        tokenizer = HashTokenizer({args.subject_string: TOK_Z, args.background_string: TOK_Y})
    else:
        if not args.tokenizer_dir:
            raise SystemExit("--tokenizer_dir (a local openai/clip-vit-large-patch14 tokenizer) is required without --synthetic")
        from transformers import CLIPTokenizer
        tokenizer = CLIPTokenizer.from_pretrained(args.tokenizer_dir)

    with torch.device("meta"):
        unet = UNetModel(**SD15_UNET_CONFIG)
        vae = AutoencoderKL(with_encoder=bool(getattr(args, "init_img", None)))
    unet, vae = unet.to_empty(device=device), vae.to_empty(device=device)
    clip_cfg = CLIPTextConfigLite(num_hidden_layers=args.synthetic_clip_layers) if args.synthetic else CLIPTextConfigLite()
    frozen = FrozenCLIPEmbedder(tokenizer=tokenizer, config=clip_cfg,
                                last_layers_skip_weights=tuple(args.clip_last_layers_skip_weights))
    arc2face = CLIPTextModelWrapper(clip_cfg)
    sbg = SubjBasisGenerator(num_out_embs_per_layer=args.num_vectors_per_subj_token, clip_tokenizer=tokenizer,
                             clip_config=clip_cfg)
    if args.synthetic:
        unet.load_state_dict(synth_state_dict(spec_of(unet), args.seed_weights))
        vae.load_state_dict(synth_state_dict(spec_of(vae), args.seed_weights + 1))
        torch.manual_seed(args.seed_weights)         # CLIP-shaped modules keep their own (HF-style) random init
    else:
        parts = split_sd15_checkpoint(torch.load(args.ckpt, map_location="cpu"))
        unet.load_state_dict(parts["unet"])
        vae.load_state_dict(parts["vae"])
        frozen.transformer.load_state_dict(parts["clip"], strict=False)
        if args.arc2face_ckpt:
            arc2face.load_state_dict(torch.load(args.arc2face_ckpt, map_location="cpu"))
        if not args.subj_ckpt:
            raise SystemExit("--subj_ckpt (state_dict of SubjBasisGenerator) is required without --synthetic")
        sbg.load_state_dict(torch.load(args.subj_ckpt, map_location="cpu"), strict=False)
    unet.eval().prepare()
    vae.eval()
    em = EmbeddingManagerLite(tokenizer, subject_strings=(args.subject_string,),
                              placeholder_tokens={args.subject_string: tokenizer.encode(args.subject_string, add_special_tokens=False)[0]},
                              token2num_vectors={args.subject_string: args.num_vectors_per_subj_token},
                              arc2face_text_encoder=arc2face,
                              zs_adaface_prompt_embs_inf_type=args.zs_adaface_prompt_embs_inf_type)
    em.string_to_subj_basis_generator_dict[args.subject_string] = sbg
    model = LatentDiffusionLite(unet, cond_stage_model=frozen, embedding_manager=em, first_stage_model=vae)
    return model.to(device).eval(), tokenizer


def expand_prompt(prompt: str, subject_string: str, n_vectors: int) -> str:
    """stable_txt2img.py / embedding_manager: the subject token is followed by n-1 commas that the splice overwrites
    ("a photo of a z, , , ..." - SURVEY.md section 8(d) config 2)."""
    words = prompt.split()
    out = []
    for w in words:
        out.append(w)
        if w.strip(",.") == subject_string:
            out.append(", " * (n_vectors - 1))
    return " ".join(out).strip()


def save_images(imgs: torch.Tensor, outdir: str, base: int, prefix: str) -> List[str]:
    """imgs: [n, 3, H, W] in [0, 1] on the host -> PNG files (stable_txt2img.py:689-700)."""
    import numpy as np
    from PIL import Image
    os.makedirs(outdir, exist_ok=True)
    paths = []
    for i, im in enumerate(imgs):
        arr = (255. * im.permute(1, 2, 0).numpy()).round().clip(0, 255).astype(np.uint8)
        p = os.path.join(outdir, f"{prefix}-{base + i:05d}.png")
        Image.fromarray(arr).save(p)
        paths.append(p)
    return paths


def save_grid(imgs: torch.Tensor, path: str, n_rows: int):
    import numpy as np
    from PIL import Image
    n, c, h, w = imgs.shape
    cols = max(1, n_rows)
    rows = (n + cols - 1) // cols
    canvas = torch.ones(c, rows * h, cols * w)
    for i in range(n):
        r, cc = divmod(i, cols)
        canvas[:, r * h:(r + 1) * h, cc * w:(cc + 1) * w] = imgs[i]
    Image.fromarray((255. * canvas.permute(1, 2, 0).numpy()).round().clip(0, 255).astype(np.uint8)).save(path)


def parse_args(argv=None):
    p = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    p.add_argument("--prompt", type=str, default="a photo of a z", help="the prompt to render")           # :41
    p.add_argument("--neg_prompt", type=str, default="", help="the negative prompt")                        # :48
    p.add_argument("--from_file", type=str, default=None, help="one prompt per line")                        # :155
    p.add_argument("--outdir", type=str, default="outputs/txt2img-samples")                                 # :64
    p.add_argument("--ddim_steps", type=int, default=50)                                                    # :86
    p.add_argument("--ddim_eta", type=float, default=0.0)                                                   # :97
    p.add_argument("--n_repeat", type=int, default=1, help="sample this often")                              # :103
    p.add_argument("--H", type=int, default=512)                                                            # :109
    p.add_argument("--W", type=int, default=512)                                                            # :115
    p.add_argument("--C", type=int, default=4)                                                              # :121
    p.add_argument("--f", type=int, default=8)                                                              # :127
    p.add_argument("--n_samples", type=int, default=4, help="images per prompt")                             # :133
    p.add_argument("--bs", type=int, default=-1, help="batch size per GPU (default: n_samples)")            # :140
    p.add_argument("--n_rows", type=int, default=0, help="columns of the grid (default: n_samples)")        # :142
    p.add_argument("--scale", type=float, nargs="+", default=[10.0, 4.0],
                   help="guidance scale, annealed from the first to the second value (one value: constant)")  # :148
    p.add_argument("--ckpt", type=str, default=None, help="SD-1.5 LatentDiffusion checkpoint")               # :166
    p.add_argument("--seed", type=int, default=42)                                                          # :172
    p.add_argument("--subj_ckpt", type=str, default=None, help="state_dict of the SubjBasisGenerator")
    p.add_argument("--arc2face_ckpt", type=str, default=None, help="state_dict of the Arc2Face CLIP text encoder")
    p.add_argument("--tokenizer_dir", type=str, default=None)
    p.add_argument("--face_embs", type=str, default=None, help=".pt file with [n, 512] ArcFace ID embeddings (--ref_images stand-in)")
    p.add_argument("--clip_last_layers_skip_weights", type=float, nargs="+", default=[1, 1])              # :235
    p.add_argument("--subject_string", type=str, default="z")                                               # :239
    p.add_argument("--background_string", type=str, default="y")                                            # :242
    p.add_argument("--num_vectors_per_subj_token", type=int, default=16)                                    # :246
    p.add_argument("--zs_adaface_prompt_embs_inf_type", type=str, default="full_half_pad")                  # :264
    p.add_argument("--zs_out_id_embs_scale_range", type=float, nargs=2, default=[1.0, 1.0])                 # :269
    p.add_argument("--no_cuda_graph", action="store_true")
    p.add_argument("--save_latents", action="store_true", help="also torch.save the latents next to the images")
    p.add_argument("--save_conditioning", action="store_true",
                   help="also torch.save the conditioning tensors (c, uc) and x_T of every batch (parity checks); "
                        "img2img: the posterior noise, the stochastic_encode noise and z_enc instead of x_T")
    p.add_argument("--init_img", type=str, default=None,
                   help="img2img: start from this image (RGB, exactly --W x --H pixels) instead of noise")
    p.add_argument("--strength", type=float, default=0.75,
                   help="img2img: noise level of the init image; t_enc = int(strength * ddim_steps) in [2, ddim_steps - 1]")
    p.add_argument("--synthetic", action="store_true", help="random-init weights + hashing tokenizer (no files needed)")
    p.add_argument("--synthetic_clip_layers", type=int, default=12)
    p.add_argument("--seed_weights", type=int, default=1234)
    args = p.parse_args(argv)
    if len(args.scale) == 1:
        args.scale = [args.scale[0], args.scale[0]]
    if len(args.scale) != 2:
        p.error("--scale takes one or two values")
    if args.W % 64 or args.H % 64 or args.f != 8:
        p.error("--H / --W must be multiples of 64 and --f 8 (the SD-1.5 VAE)")
    if not args.synthetic and not args.ckpt:
        p.error("--ckpt is required unless --synthetic is given")
    if args.init_img:
        from .ddim import img2img_t_enc
        try:
            img2img_t_enc(args.strength, args.ddim_steps)
        except ValueError as e:
            p.error(str(e))
    return args


def load_init_image(path: str, H: int, W: int) -> torch.Tensor:
    """SD scripts/img2img.py load_img: RGB -> [1, 3, H, W] fp32 in [-1, 1]; the size must already be W x H."""
    import numpy as np
    from PIL import Image
    image = Image.open(path).convert("RGB")
    if image.size != (W, H):
        raise SystemExit(f"--init_img {path} is {image.size[0]}x{image.size[1]} pixels; --W x --H is {W}x{H}")
    arr = np.array(image).astype(np.float32) / 255.0
    return 2. * torch.from_numpy(arr[None].transpose(0, 3, 1, 2).copy()) - 1.


@torch.no_grad()
def run(args) -> List[str]:
    import torch.distributed as dist
    from .ddim import DDIMSampler
    from .parallel_sampling import shard_range

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("txt2img: no CUDA device - the B200 path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=device)

    model, _ = build_pipeline(args, device)
    sampler = DDIMSampler(model, use_cuda_graph=not args.no_cuda_graph)
    n_vec = args.num_vectors_per_subj_token
    if args.from_file:
        with open(args.from_file) as f:
            prompts = [ln.strip() for ln in f if ln.strip()]
    else:
        prompts = [args.prompt]
    # work items = (prompt, repeat, sample): sharded contiguously over the ranks (SURVEY.md section 8(e))
    items = [(pi, r, s) for pi in range(len(prompts)) for r in range(args.n_repeat) for s in range(args.n_samples)]
    b0, b1 = shard_range(len(items), world, rank)
    mine = items[b0:b1]
    bs = args.bs if args.bs > 0 else args.n_samples

    if args.face_embs:
        id_embs = torch.load(args.face_embs, map_location="cpu").float().reshape(-1, 512)[:1].to(device)
    else:
        id_embs = torch.randn(1, 512, generator=torch.Generator().manual_seed(args.seed)).to(device)
    id_embs = torch.nn.functional.normalize(id_embs, p=2, dim=-1)                                  # adaface/util.py:311
    shape = [args.C, args.H // args.f, args.W // args.f]
    init_image = t_enc = None
    if args.init_img:
        from .ddim import img2img_t_enc
        t_enc = img2img_t_enc(args.strength, args.ddim_steps)
        init_image = load_init_image(args.init_img, args.H, args.W).to(device)
        sampler.make_schedule(ddim_num_steps=args.ddim_steps, ddim_eta=args.ddim_eta, verbose=False)
    paths, all_imgs = [], []
    for start in range(0, len(mine), bs):
        chunk = mine[start:start + bs]
        n = len(chunk)
        texts = [expand_prompt(prompts[pi], args.subject_string, n_vec) for pi, _, _ in chunk]
        c = model.get_learned_conditioning(texts, zs_clip_features=None, zs_id_embs=id_embs,
                                           zs_out_id_embs_scale_range=tuple(args.zs_out_id_embs_scale_range))   # :606-613
        uc = model.get_learned_conditioning([args.neg_prompt] * n)                                              # :602
        if init_image is None:
            g = torch.Generator().manual_seed(args.seed + 1000 * rank + start)
            x_T = torch.randn(n, *shape, generator=g).to(device)                                                # :578
            samples, _ = sampler.sample(S=args.ddim_steps, batch_size=n, shape=shape, conditioning=c,
                                        unconditional_conditioning=uc, guidance_scale=tuple(args.scale),
                                        eta=args.ddim_eta, x_T=x_T, verbose=False)                              # :614-626
            saved = {"x_T": x_T.cpu()}
        else:
            # img2img.py: encode the batch of init images, noise to t_enc, decode with CFG.  The two noises are drawn
            # where the reference draws them (posterior: host generator; stochastic_encode: randn_like on the device)
            torch.manual_seed(args.seed + 1000 * rank + start)
            posterior = model.encode_first_stage(init_image.repeat(n, 1, 1, 1))
            post_noise = torch.randn(posterior.mean.shape)
            init_latent = posterior.scaled_sample(model.scale_factor, noise=post_noise)    # get_first_stage_encoding
            se_noise = torch.randn_like(init_latent)
            z_enc = sampler.stochastic_encode(init_latent, torch.full((n,), t_enc, dtype=torch.long, device=device),
                                              noise=se_noise)
            samples = sampler.decode(z_enc, c, t_enc, guidance_scale=args.scale[0], unconditional_conditioning=uc)
            saved = {"posterior_noise": post_noise, "stochastic_encode_noise": se_noise.cpu(), "z_enc": z_enc.cpu(),
                     "t_enc": t_enc}
        x = model.decode_first_stage(samples)                                                                   # :685
        x = torch.clamp((x + 1.0) / 2.0, min=0.0, max=1.0).cpu()                                                # :687
        paths += save_images(x, os.path.join(args.outdir, "samples"), b0 + start, f"r{rank}")
        all_imgs.append(x)
        if args.save_latents:
            torch.save(samples.cpu(), os.path.join(args.outdir, "samples", f"r{rank}-{b0 + start:05d}-latents.pt"))
        if args.save_conditioning:
            torch.save({"c": c[0].cpu(), "uc": uc[0].cpu(), "prompts": texts, **saved},
                       os.path.join(args.outdir, "samples", f"r{rank}-{b0 + start:05d}-cond.pt"))
    if all_imgs:
        save_grid(torch.cat(all_imgs), os.path.join(args.outdir, f"grid-r{rank}.png"), args.n_rows or args.n_samples)
    if world > 1:
        dist.barrier()
    if rank == 0:
        print(f"txt2img: {len(items)} image(s) over {world} GPU(s) -> {args.outdir}")
    return paths


def main(argv=None):
    args = parse_args(argv)
    run(args)


if __name__ == "__main__":
    main(sys.argv[1:])
