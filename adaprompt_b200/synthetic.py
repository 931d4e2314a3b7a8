"""Random-init / synthetic-data builders shared by bench.py, scripts/bench_train.py and the GPU tests: the Stage-1
distillation stack of BASELINE.json configs[3] (there is no network for real checkpoints or a tokenizer vocabulary)."""
from __future__ import annotations

import types

import torch


class StubTokenizer:
    """The handful of CLIP token ids the AdaFace prompts use (ids from SURVEY.md section 8(c))."""
    pad_token_id = 49407
    vocab = {"photo": 1125, "of": 539, "a": 320, "id": 1014, "person": 2533, ",": 267, "z": 345}

    def _ids(self, text):
        return [self.vocab[w] for w in text.replace(",", " , ").split()]

    def encode(self, text, add_special_tokens=False):
        return self._ids(text)

    def __call__(self, text, truncation=True, padding="max_length", max_length=77, return_tensors="pt", **kw):
        texts = [text] if isinstance(text, str) else list(text)
        rows = [([49406] + self._ids(t) + [49407] * max_length)[:max_length] for t in texts]
        return types.SimpleNamespace(input_ids=torch.tensor(rows))


def stage1_stack(dev, unet=None):
    """-> (DistillStep, trainable parameter list): frozen SD-1.5 UNet (seed 1234), trainable SubjBasisGenerator
    (12-layer CLIP text model), frozen CLIP embedder and Arc2Face text encoder, all random-init."""
    from .clip_text import CLIPTextModelWrapper
    from .ldm_lite import SD15_UNET_CONFIG
    from .subj_basis_generator import SubjBasisGenerator
    from .train_cond import DistillStep, trainable_parameters
    from .unet import UNetModel
    from .weights import spec_of, synth_state_dict
    if unet is None:
        with torch.device("meta"):
            unet = UNetModel(**SD15_UNET_CONFIG)
        unet = unet.to_empty(device=dev)
        unet.load_state_dict(synth_state_dict(spec_of(unet), 1234))
        unet.eval().prepare()
    for p in unet.parameters():
        p.requires_grad = False

    def clip(seed, train):
        m = CLIPTextModelWrapper().to(dev)
        sd = synth_state_dict({k: tuple(v.shape) for k, v in m.state_dict().items()}, seed)
        for k in sd:
            if "embedding" in k:
                sd[k] = torch.randn(sd[k].shape, generator=torch.Generator().manual_seed(seed)) * 0.02
        m.load_state_dict(sd)
        for p in m.parameters():
            p.requires_grad = train
        return m

    tok = StubTokenizer()
    sbg = SubjBasisGenerator(num_out_embs_per_layer=16, clip_tokenizer=tok)
    sbg.prompt2token_proj = clip(41, True)
    sbg = sbg.to(dev).train()
    frozen, arc2face = clip(42, False), clip(43, False).eval()
    frozen.text_model.last_layers_skip_weights = [0.5, 0.5]
    acp = torch.linspace(0.9991, 0.0047, 1000)
    step = DistillStep(unet, frozen.text_model, sbg, arc2face, tok, acp, 345)
    return step, trainable_parameters(sbg)


def stage1_batch(dev, bs: int, latent: int, generator: torch.Generator, masks: bool = False):
    """One synthetic micro-batch: x0 / noise / t / a fixed teacher eps (the diffusers teacher is unavailable, SURVEY.md
    section 8(d) config 4) / L2-normalised 512-d ArcFace embeddings / the tokens of "a photo of a z, , ...".
    masks: also "img_mask" and "fg_mask" (float [bs, 1, H, H]) drawn after everything else, so the other tensors are
    those of masks=False: see synthetic_masks."""
    g, H = generator, latent
    prompt = [49406, 320, 1125, 539, 320, 345] + [267] * 15 + [49407] * 56
    batch = {"x0": torch.randn(bs, 4, H, H, generator=g).to(dev), "noise": torch.randn(bs, 4, H, H, generator=g).to(dev),
             "t": torch.randint(0, 1000, (bs,), generator=g).to(dev),
             "teacher_eps": torch.randn(bs, 4, H, H, generator=g).to(dev),
             "face_embs": torch.nn.functional.normalize(torch.randn(bs, 512, generator=g), dim=-1).to(dev),
             "tokens": torch.tensor([prompt] * bs).to(dev)}
    if masks:
        img_mask, fg_mask = synthetic_masks(bs, H, g)
        batch["img_mask"], batch["fg_mask"] = img_mask.to(dev), fg_mask.to(dev)
    return batch


def synthetic_masks(bs: int, H: int, generator: torch.Generator):
    """Plausible masks of a face-image batch at latent size H x H (CPU, float [bs, 1, H, H]):
      img_mask: the image inside a zero border of 0 .. H/8 pixels on each side (augmentation padding);
      fg_mask:  a face box of 3/8 .. 5/8 of the side, placed inside the image."""
    g = generator
    img = torch.zeros(bs, 1, H, H)
    fg = torch.zeros(bs, 1, H, H)
    for b in range(bs):
        t, bo, l, r = (int(v) for v in torch.randint(0, H // 8 + 1, (4,), generator=g))
        img[b, :, t:H - bo, l:H - r] = 1
        side = int(torch.randint(3 * H // 8, 5 * H // 8 + 1, (1,), generator=g))
        y0 = t + int(torch.randint(0, max(1, H - bo - t - side + 1), (1,), generator=g))
        x0 = l + int(torch.randint(0, max(1, H - r - l - side + 1), (1,), generator=g))
        fg[b, :, y0:y0 + side, x0:x0 + side] = 1
    return img, fg * img
