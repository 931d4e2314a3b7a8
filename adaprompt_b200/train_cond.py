"""Stage-1 distillation step, conditioning half and step driver (SURVEY.md section 8 row T1, configs[3]).

Gradient path of the reference (ldm/models/diffusion/ddpm.py):
  loss (:3010-3037) -> UNet (frozen, train.py) -> layerwise context c [16B,77,768]
       -> FrozenCLIPEmbedder (frozen weights, ldm/modules/encoders/modules.py:260-283,361-370)
       -> EmbeddingManager splice (embedding_manager.py:1516-1562; rows of the 16 ID tokens)
       -> SubjBasisGenerator.forward (adaface/subj_basis_generator.py:470-567, is_training=True):
          prompt2token_proj = a TRAINABLE CLIP text model (arc2face_models.py:178-280) + hidden_state_layer_weights
          (grad scaler 5, :498,:580) + prompt2token_proj_grad_scaler (:528-529).
Data parallel: one process per GPU, one all-reduce (mean) of the SubjBasisGenerator gradients per optimizer step in a
single flat fp32 bucket over NCCL / NVLink (main.py:829 uses Lightning DDP for the same exchange).

As in train.py, torch.autograd is the tape; the arithmetic of every layer is a C-ABI kernel.  Index plumbing
(embedding-row gather / scatter, the x16 layer repeat, concatenations) uses torch tensor ops.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence

import torch
from torch.autograd import Function

from . import ops
from .adaface_util import _ScaleGradFn, _tokenize, arc2face_forward_face_embs
from .clip_text import CLIPEncoderLayer, CLIPTextTransformer
from .train import LayerNormFn, calc_recon_loss, check_image_mask, distill_loss, linear, unet_forward_train

N_CA_LAYERS = 16


def grad_scale(x, alpha):
    """gen_gradient_scaler (adaface/util.py:60-72): alpha 1 -> identity, 0 -> detach."""
    if alpha == 1:
        return x
    if alpha == 0:
        return x.detach()
    return _ScaleGradFn.apply(x, alpha)


class QuickGeluFn(Function):
    @staticmethod
    def forward(ctx, x):
        ctx.save_for_backward(x)
        return ops.quick_gelu(x)

    @staticmethod
    def backward(ctx, dy):
        (x,) = ctx.saved_tensors
        return ops.quick_gelu(x, dy.contiguous())


class AttnSmallFn(Function):
    """CLIP text self-attention (77 tokens, causal, MKV aware): qkv bf16 [B*L, E*(1+2m)] -> bf16 [B*L, E]."""

    @staticmethod
    def forward(ctx, qkv, B, heads, L, E, m, scale):
        o = torch.empty(B * L, E, dtype=torch.bfloat16, device=qkv.device)
        ops.attention_small(qkv, o, B=B, heads=heads, L=L, k_off=E, v_off=E + E * m, mult=m, scale=scale, causal=True)
        ctx.save_for_backward(qkv)
        ctx.geom = (B, heads, L, E, m, scale)
        return o

    @staticmethod
    def backward(ctx, do):
        (qkv,) = ctx.saved_tensors
        B, heads, L, E, m, scale = ctx.geom
        dqkv = ops.attention_small_bwd(qkv, do.contiguous(), B=B, heads=heads, L=L, k_off=E, v_off=E + E * m, mult=m,
                                       scale=scale, causal=True)
        return dqkv, None, None, None, None, None, None


class SpliceRowsFn(Function):
    """EmbeddingManager row replacement (embedding_manager.py:1516-1562): dst[r, first[r]+k] = src[src_index[r], k].
    dst carries no gradient of its own rows that were overwritten; src gets the gathered rows back."""

    @staticmethod
    def forward(ctx, dst, src, first, src_index):
        out = dst.clone()
        ops.splice_rows(out, src.contiguous(), first, src_index)
        ctx.save_for_backward(first, src_index)
        ctx.src_shape = src.shape
        return out

    @staticmethod
    def backward(ctx, g):
        # no data-dependent shapes (torch.nonzero would synchronise the host and break CUDA-graph capture): rows without
        # the placeholder (first < 0) and positions past the sequence end contribute zeros / keep their gradient
        first, src_index = ctx.saved_tensors
        S, K, D = ctx.src_shape
        R, N = g.shape[0], g.shape[1]
        pos = first.long().clamp_min(0)[:, None] + torch.arange(K, device=g.device)[None]            # [R, K]
        valid = ((first >= 0)[:, None] & (pos < N))[..., None]                                      # [R, K, 1]
        idx = pos.clamp_max(N - 1)[..., None].expand(R, K, D)
        picked = g.gather(1, idx)                                                                   # [R, K, D]
        dsrc = torch.zeros(S, K, D, dtype=g.dtype, device=g.device)
        dsrc.index_add_(0, src_index.long(), torch.where(valid, picked, torch.zeros_like(picked)))
        dd = g.scatter(1, idx, torch.where(valid, torch.zeros_like(picked), picked))
        return dd, dsrc, None, None


# ------------------------------------------------------------------------------------------------ CLIP text layers
def _kv_rows(w, m, H, hd):
    # reference key order (arc2face_models.py:117-131) -> kernel order [head][r][hd]; same as CLIPEncoderLayer._pack
    return w.reshape(m, H, hd, *w.shape[1:]).transpose(0, 1).reshape(m * H * hd, *w.shape[1:])


def _bf16_pair(w: torch.Tensor):
    wb = w.detach().to(torch.bfloat16).contiguous()
    return wb, wb.t().contiguous()


def _layer_weights(layer: CLIPEncoderLayer, trainable: bool) -> dict:
    """fp32 (weight, bias) views in kernel layout + bf16 operand packs.  Trainable layers rebuild them every step (the
    weights move); frozen layers cache them."""
    if not trainable:
        c = layer.__dict__.get("_train_pk")
        if c is not None:
            return c
    a = layer.self_attn
    E, H, hd = a.embed_dim, a.num_heads, a.head_dim
    m = a.k_proj.weight.shape[0] // E
    wqkv = torch.cat([a.q_proj.weight, _kv_rows(a.k_proj.weight, m, H, hd), _kv_rows(a.v_proj.weight, m, H, hd)], 0)
    bqkv = torch.cat([a.q_proj.bias, _kv_rows(a.k_proj.bias, m, H, hd), _kv_rows(a.v_proj.bias, m, H, hd)], 0)
    out = {"m": m}
    for name, (w, b) in {"qkv": (wqkv, bqkv), "o": (a.out_proj.weight, a.out_proj.bias),
                         "fc1": (layer.mlp.fc1.weight, layer.mlp.fc1.bias),
                         "fc2": (layer.mlp.fc2.weight, layer.mlp.fc2.bias)}.items():
        wb, wt = _bf16_pair(w)
        out[name] = (wb, wt, b.detach().float().contiguous(), w if trainable else None, b if trainable else None)
    if not trainable:
        layer.__dict__["_train_pk"] = out
    return out


def _lin(x, pk, residual=None, out_dtype=torch.float32):
    wb, wt, b, wp, bp = pk
    return linear(x, wb, wt, b, residual=residual, out_dtype=out_dtype, w_param=wp, b_param=bp)


def clip_layer_train(layer: CLIPEncoderLayer, h: torch.Tensor, B: int, L: int, trainable: bool) -> torch.Tensor:
    """HF CLIPEncoderLayer as CLIPEncoderLayer._run, with grad.  h fp32 [B*L, E]."""
    a = layer.self_attn
    E, H = a.embed_dim, a.num_heads
    pk = _layer_weights(layer, trainable)
    ln1, ln2 = layer.layer_norm1, layer.layer_norm2
    p = (lambda t: t) if trainable else (lambda t: t.detach())
    x = LayerNormFn.apply(h, p(ln1.weight), p(ln1.bias), float(ln1.eps), torch.bfloat16)
    qkv = _lin(x, pk["qkv"], out_dtype=torch.bfloat16)
    o = AttnSmallFn.apply(qkv, B, H, L, E, pk["m"], a.scale)
    h1 = _lin(o, pk["o"], residual=h)
    x2 = LayerNormFn.apply(h1, p(ln2.weight), p(ln2.bias), float(ln2.eps), torch.bfloat16)
    u = QuickGeluFn.apply(_lin(x2, pk["fc1"], out_dtype=torch.bfloat16))
    return _lin(u, pk["fc2"], residual=h1)


def clip_encode_train(tm: CLIPTextTransformer, h: torch.Tensor, layer_weights, trainable: bool) -> torch.Tensor:
    """CLIPTextTransformer.encode with grad.  h fp32 [B, L, E] (token + position embeddings); layer_weights: None, a
    sequence of already-normalised floats, or a tensor [n, 1] (normalised here, arc2face_models.py:236-246) that may
    require grad.  Returns the final-LayerNormed fp32 [B, L, E]."""
    B, L, E = h.shape
    x = h.reshape(B * L, E).contiguous()
    states = [x]
    for layer in tm.encoder.layers:
        x = clip_layer_train(layer, x, B, L, trainable)
        states.append(x)
    if layer_weights is None:
        mixed = states[-1]
    else:
        if torch.is_tensor(layer_weights):
            w = layer_weights.reshape(-1)
            w = w / w.sum()
        else:
            w = [float(v) for v in layer_weights]
        n = len(w)
        mixed = sum(w[i] * states[len(states) - n + i] for i in range(n))
    ln = tm.final_layer_norm
    p = (lambda t: t) if trainable else (lambda t: t.detach())
    out = LayerNormFn.apply(mixed, p(ln.weight), p(ln.bias), float(ln.eps), torch.float32)
    return out.reshape(B, L, E)


# ------------------------------------------------------------------------------------------------ SubjBasisGenerator
def sbg_forward_train(sbg, arc2face_id_embs: torch.Tensor, out_id_embs_scale: float = 1.0):
    """SubjBasisGenerator.forward(is_training=True), face branch (subj_basis_generator.py:470-567), with grad w.r.t.
    prompt2token_proj and hidden_state_layer_weights.  -> (adaface_subj_embs [BS,L,16,768], adaface_prompt_embs)."""
    tm = sbg.prompt2token_proj.text_model
    dev = arc2face_id_embs.device
    BS = arc2face_id_embs.shape[0]
    trainable = sbg.prompt2token_proj_grad_scale != 0
    hw = sbg.hidden_state_layer_weights
    if hw is not None:
        hw = grad_scale(hw, 5)                                                                      # :498,:580
    if sbg.pad_embeddings is None:
        sbg.generate_pad_embeddings()
    pad_embeddings = sbg.pad_embeddings.to(dev)
    template = ["photo of a " + ", " * 16 for _ in range(BS)]                                      # adaface/util.py:165
    input_ids = _tokenize(sbg.clip_tokenizer, template, 77, dev)
    emb = tm.embeddings
    tok_w = emb.token_embedding.weight if trainable else emb.token_embedding.weight.detach()
    pos_w = emb.position_embedding.weight if trainable else emb.position_embedding.weight.detach()
    tok = tok_w[input_ids]                                                                          # gather (+ scatter-add backward)
    tok = torch.cat([tok[:, :4], arc2face_id_embs.float(), tok[:, 20:]], dim=1)                     # adaface/util.py:184
    h = tok + pos_w[None, :77]
    with torch.set_grad_enabled(trainable and torch.is_grad_enabled()):
        prompt_embeds = clip_encode_train(tm, h, hw, trainable)                                     # arc2face_models.py:204-248
    core = prompt_embeds[:, 4:20]
    full_pad = torch.cat([prompt_embeds[:, :22], pad_embeddings[22:-1].expand(BS, -1, -1), prompt_embeds[:, -1:]], 1)
    full_pad = grad_scale(full_pad, sbg.prompt2token_proj_grad_scale)                               # :528-529
    core = grad_scale(core, sbg.prompt2token_proj_grad_scale)
    subj = core.unsqueeze(1).repeat(1, sbg.num_out_layers, 1, 1)                                    # :558
    if out_id_embs_scale != 1:
        pe = pad_embeddings[4:4 + sbg.num_out_embs_per_layer].unsqueeze(0).unsqueeze(0)
        subj = subj * out_id_embs_scale + pe * (1 - out_id_embs_scale)
    return subj, full_pad


def conditioning_train(frozen_tm: CLIPTextTransformer, tokens: torch.Tensor, adaface_subj_embs: torch.Tensor,
                       placeholder_token: int, K: int = 16, dedup: bool = True,
                       layers_identical: Optional[bool] = None, groups: int = 1) -> torch.Tensor:
    """EmbeddingManager.forward + FrozenCLIPEmbedder with grad w.r.t. adaface_subj_embs [BS, 16, K, 768].
    tokens int64 [B, 77] -> c fp32 [16*B, 77, 768] (layer index minor to batch, embedding_manager.py:1349-1353).
    dedup: encode one of the 16 layer copies when they are identical (always true for the face branch, :558);
    layers_identical: what the caller knows about that by construction (None: compare on the device - one host read).
    No host synchronisation otherwise: the i-th prompt that holds the placeholder takes subject i mod BS (the
    reference's repeat to the number of occurrences, :1449-1451), prompts without it pass through the splice.
    groups: the rows are `groups` independent forward calls stacked along the batch (the micro-batches of an optimizer
    step): occurrences are counted, and subjects assigned, within each group of B / groups prompts and BS / groups
    subjects - exactly what `groups` separate calls would do."""
    B, N = tokens.shape
    L = N_CA_LAYERS
    tw = frozen_tm.embeddings.token_embedding.weight.detach().float().contiguous()
    pos = frozen_tm.embeddings.position_embedding.weight.detach().float()
    emb = ops.gather_rows(tw, tokens.contiguous())                                                 # [B, N, 768]
    first_b = ops.find_first_token(tokens.contiguous(), placeholder_token)                         # [B]
    has = first_b >= 0
    BS = adaface_subj_embs.shape[0]
    identical = dedup and adaface_subj_embs.shape[1] == L
    if identical:
        if layers_identical is None:
            with torch.no_grad():
                identical = bool((adaface_subj_embs == adaface_subj_embs[:, :1]).all().item())
        else:
            identical = bool(layers_identical)
    w = frozen_tm.last_layers_skip_weights
    if B % groups or BS % groups:
        raise ValueError("conditioning_train: batch / subjects not divisible into `groups` calls")

    def occurrence_index(has_rows: torch.Tensor, n_src: int) -> torch.Tensor:
        """row -> index of the subject it takes: the i-th occurrence inside its group takes the group's subject i mod n."""
        hg = has_rows.view(groups, -1).int()
        rank = (torch.cumsum(hg, 1) - 1).clamp_min(0)
        per = n_src // groups
        base = torch.arange(groups, device=has_rows.device, dtype=rank.dtype)[:, None] * per
        return (rank % per + base).reshape(-1).to(torch.int32).contiguous()

    if identical:
        src = adaface_subj_embs[:, 0, :K].contiguous()                                             # [BS, K, 768]
        src_index = occurrence_index(has, BS)
        spliced = SpliceRowsFn.apply(emb, src, first_b, src_index)
        z = clip_encode_train(frozen_tm, spliced + pos[None, :N], w, trainable=False)
        return z.unsqueeze(1).expand(B, L, N, z.shape[-1]).reshape(B * L, N, z.shape[-1])
    emb16 = emb.unsqueeze(1).repeat(1, L, 1, 1).view(B * L, N, -1)
    first16 = first_b.repeat_interleave(L).contiguous()
    has16 = first16 >= 0
    src = adaface_subj_embs.reshape(BS * adaface_subj_embs.shape[1], *adaface_subj_embs.shape[2:])[:, :K].contiguous()
    src_index = occurrence_index(has16, src.shape[0])
    spliced = SpliceRowsFn.apply(emb16, src, first16, src_index)
    return clip_encode_train(frozen_tm, spliced + pos[None, :N], w, trainable=False)


# ------------------------------------------------------------------------------------------------ step driver
def trainable_parameters(sbg) -> List[torch.nn.Parameter]:
    return [p for p in sbg.parameters() if p.requires_grad]


class GradBucket:
    """The gradients of a FIXED trainable-parameter list as one flat fp32 buffer; every p.grad is a view of it.

    * autograd accumulates micro-batch gradients straight into the bucket (no torch.cat, no copy-back);
    * a parameter that got no gradient on this rank contributes zeros - the bucket has the same size on every rank,
      which a collective needs (ranks with different sets of touched parameters would otherwise hang NCCL);
    * the one data-path collective of the step (SURVEY.md section 8(e)) is a single all-reduce of the bucket (NCCL over
      NVLink / NVSwitch on GPUs, gloo in the CPU tests), SUM scaled to the mean (main.py:829 uses Lightning DDP);
    * clipping by norm (ddpm.py:607, gradient_clip_val 0.5) is two kernels on the bucket and no host synchronisation;
    * Prodigy.step consumes the bucket as it is."""

    def __init__(self, params: Sequence[torch.nn.Parameter]):
        self.params = list(params)
        if not self.params:
            raise ValueError("GradBucket: empty parameter list")
        from .prodigy import flat_layout
        dev = self.params[0].device
        offs, total = flat_layout(self.params)      # same layout as Prodigy's parameter / state buckets (aligned starts)
        self.flat = torch.zeros(total, dtype=torch.float32, device=dev)
        self.views = [self.flat[o:o + p.numel()].view(p.shape) for p, o in zip(self.params, offs)]
        self._work = None

    def begin_step(self):
        """Zero the bucket and (re-)bind p.grad to its views (an optimizer may have set them to None)."""
        self.flat.zero_()
        for p, v in zip(self.params, self.views):
            if p.dtype != torch.float32:
                raise TypeError("GradBucket: trainable parameters must be fp32")
            p.grad = v

    def allreduce(self, world_size: int, group=None, async_op: bool = False):
        import torch.distributed as dist
        if world_size <= 1:
            return None
        self._work = dist.all_reduce(self.flat, op=dist.ReduceOp.SUM, group=group, async_op=async_op)
        self._scale = 1.0 / world_size
        if not async_op:
            self.wait()
        return self._work

    def wait(self):
        if self._work is not None:
            self._work.wait()
        self._work = None
        if getattr(self, "_scale", None) is not None:
            self.flat.mul_(self._scale)
            self._scale = None

    def clip_(self, max_norm: float = 0.5) -> torch.Tensor:
        """In-place clip by total norm; returns the norm before clipping as a 0-d tensor (no host sync)."""
        total = torch.linalg.vector_norm(self.flat)
        self.flat.mul_(torch.clamp(max_norm / (total + 1e-6), max=1.0))
        return total


def allreduce_gradients(params: Sequence[torch.nn.Parameter], world_size: int, group=None) -> Optional[torch.Tensor]:
    """Functional form over ad-hoc p.grad tensors: builds the fixed-size bucket (zeros where p.grad is None), all-reduces
    it to the mean and writes the result back to every p.grad.  Returns the bucket."""
    params = list(params)
    if not params:
        return None
    grads = [p.grad for p in params]
    bucket = GradBucket(params)
    bucket.begin_step()
    for v, g in zip(bucket.views, grads):
        if g is not None:
            v.copy_(g)
    bucket.allreduce(world_size, group=group)
    return bucket.flat


def clip_grad_norm(params: Sequence[torch.nn.Parameter], max_norm: float = 0.5) -> float:
    """gradient_clip_val 0.5 by norm (ddpm.py:607 / Lightning trainer) over p.grad; one norm kernel per tensor but a
    single host read."""
    grads = [p.grad for p in params if p.grad is not None]
    if not grads:
        return 0.0
    total = torch.linalg.vector_norm(torch.stack([torch.linalg.vector_norm(g.float()) for g in grads]))
    scale = torch.clamp(max_norm / (total + 1e-6), max=1.0)
    for g in grads:
        g.mul_(scale.to(g.dtype))
    return float(total)


class _QSampleOnly:
    """The two things Arc2FaceTeacher.forward reads from the LatentDiffusion object (ddpm.py:5448,5456)."""

    def __init__(self, alphas_cumprod: torch.Tensor):
        self.alphas_cumprod = alphas_cumprod

    def q_sample(self, x0, t, noise):
        a = self.alphas_cumprod[t].view(-1, 1, 1, 1)
        return a.sqrt() * x0 + (1 - a).sqrt() * noise


MASK_KEYS = ("img_mask", "fg_mask")


def batch_masks(batch: Dict[str, torch.Tensor]):
    """-> (img_mask, fg_mask) of a micro-batch, each None or a float / bool [B, 1, H, W] matching batch["x0"]
    (ValueError otherwise)."""
    out = []
    for k in MASK_KEYS:
        m = batch.get(k)
        if m is not None:
            check_image_mask(m, batch["x0"], f'batch["{k}"]')
        out.append(m)
    return tuple(out)


def check_mask_presence(batches: Sequence[Dict[str, torch.Tensor]]) -> None:
    """The micro-batches of one optimizer step must carry the same masks (one capture serves them all)."""
    present = [tuple(b.get(k) is not None for k in MASK_KEYS) for b in batches]
    if any(p != present[0] for p in present):
        raise ValueError(f"the micro-batches of one optimizer step disagree on which of {MASK_KEYS} they carry: {present}")


class DistillStep:
    """One Stage-1 zero-shot distillation micro-step (ddpm.py:2953-3039 with num_denoising_steps = 1):
    x_noisy = sqrt(a_t) x0 + sqrt(1 - a_t) noise (:416-419) -> student UNet with the AdaFace prompt ->
    MSE against the teacher's noise prediction.  The teacher's eps is either an input (`teacher_eps` in the batch) or
    computed by `teacher` = arc2face_teacher.Arc2FaceTeacher (ddpm.py:5402-5478, SURVEY.md section 8(f) N4) on the
    21-token Arc2Face ID prompt (ddpm.py:5427) when the batch carries none.
    A batch of real images may carry "img_mask" (latent pixels that hold image rather than padding) and "fg_mask" (the
    face), float or bool [B, 1, H, W] at the latent's resolution.  img_mask masks the student UNet's self-attention keys
    (the teacher is unchanged), and with either mask the loss is calc_recon_loss with fg_pixel_weight /
    bg_pixel_weight; without masks it is distill_loss, as before."""

    def __init__(self, unet, frozen_tm: CLIPTextTransformer, sbg, arc2face_text_encoder, tokenizer, alphas_cumprod,
                 placeholder_token: int, extra_info: Optional[dict] = None, teacher=None, fg_pixel_weight: float = 1.,
                 bg_pixel_weight: float = 1.):
        self.teacher = teacher
        self.fg_pixel_weight, self.bg_pixel_weight = fg_pixel_weight, bg_pixel_weight
        self.unet, self.frozen_tm, self.sbg = unet, frozen_tm, sbg
        self.arc2face, self.tokenizer = arc2face_text_encoder, tokenizer
        self.acp = torch.as_tensor(alphas_cumprod, dtype=torch.float32)
        self._acp_dev = {}
        self.placeholder_token = placeholder_token
        self.extra_info = dict(extra_info or {"use_layerwise_context": True, "use_conv_attn_kernel_size": -1,
                                              "placeholder2indices": None, "is_training": True})

    def _acp(self, device) -> torch.Tensor:
        a = self._acp_dev.get(device)
        if a is None:                      # one upload: a pageable host-to-device copy synchronises the stream every time
            a = self._acp_dev[device] = self.acp.to(device)
        return a

    def q_sample(self, x0, t, noise):
        a = self._acp(x0.device)[t].view(-1, 1, 1, 1)
        return a.sqrt() * x0 + (1 - a).sqrt() * noise

    def context(self, face_embs: torch.Tensor, tokens: torch.Tensor, groups: int = 1) -> torch.Tensor:
        """groups > 1: the rows are that many micro-batches stacked along the batch (GraphedAccumStep)."""
        with torch.no_grad():
            _, id_embs = arc2face_forward_face_embs(self.tokenizer, self.arc2face, face_embs)     # embedding_manager.py:1424
        subj, _ = sbg_forward_train(self.sbg, id_embs)       # 16 identical layer copies by construction (:558)
        return conditioning_train(self.frozen_tm, tokens, subj, self.placeholder_token, layers_identical=True,
                                  groups=groups)

    @torch.no_grad()
    def teacher_eps(self, x0, t, noise, face_embs) -> torch.Tensor:
        """ddpm.py:2953-3002 with num_denoising_steps = 1: the teacher denoises the same x_noisy, conditioned on the
        Arc2Face ID prompt embeddings with all padding removed (input_max_length = 21)."""
        if self.teacher is None:
            raise RuntimeError("DistillStep: the batch has no teacher_eps and no teacher model was given")
        prompt_embs, _ = arc2face_forward_face_embs(self.tokenizer, self.arc2face, face_embs, input_max_length=21,
                                                    return_full_and_core_embs=True)
        ddpm = _QSampleOnly(self._acp(x0.device))
        preds, _, _, _ = self.teacher(ddpm, x0, noise, t, prompt_embs, num_denoising_steps=1)
        return preds[0]

    def student_extra_info(self, img_mask=None) -> dict:
        extra = dict(self.extra_info)
        if img_mask is not None:
            extra["img_mask"] = img_mask
        return extra

    def recon_loss(self, eps, target, img_mask=None, fg_mask=None) -> torch.Tensor:
        """distill_loss without masks (bit-identical to the unmasked step), calc_recon_loss with them."""
        if img_mask is None and fg_mask is None:
            return distill_loss(eps, target)
        return calc_recon_loss(eps, target, img_mask, fg_mask, self.fg_pixel_weight, self.bg_pixel_weight)

    def graphed(self):
        from .train import GraphedUNetLoss
        return self.__dict__.setdefault("_graphed", GraphedUNetLoss(self.unet, self.extra_info, self.fg_pixel_weight,
                                                                    self.bg_pixel_weight))

    def loss(self, x0, t, noise, teacher_eps, face_embs, tokens, img_mask=None, fg_mask=None) -> torch.Tensor:
        for name, m in (("img_mask", img_mask), ("fg_mask", fg_mask)):
            if m is not None:
                check_image_mask(m, x0, name)
        if teacher_eps is None:
            teacher_eps = self.teacher_eps(x0, t, noise, face_embs)
        c = self.context(face_embs, tokens)
        eps = unet_forward_train(self.unet, self.q_sample(x0, t, noise), t, c, self.student_extra_info(img_mask))
        return self.recon_loss(eps, teacher_eps, img_mask, fg_mask)

    def multi_step_backward(self, batch: Dict[str, torch.Tensor], num_denoising_steps: int, accum: int = 1,
                            use_graph: bool = False) -> torch.Tensor:
        """Student multi-step distillation (ddpm.py:2953-3039 with iter_flags['num_denoising_steps'] > 1 and
        use_arc2face_as_target): the teacher denoises num_denoising_steps times from progressively earlier timesteps
        (Arc2FaceWrapper.forward :5431-5480); for every step s that fits the accumulation budget
        (MAX_ACCUMU_BATCH_SIZE = 7: loss_start_step = max(0, ND - 7 // batch), :2967-2968) the student denoises
        q_sample(pred_x0s[s-1], ts[s], noises[s]) with grad and is matched to the teacher's noise prediction of that step;
        loss = sum_s MSE_s / sqrt(ND) (:3037).  The reference indexes `arc2face_pred_x0s[s-1]` also for s = 0, i.e. the
        first student step starts from the teacher's LAST predicted x0 (:2987) - kept, it is what the trainer computes.
        loss / accum is backpropagated into the trainable parameters' .grad; returns the detached loss."""
        if self.teacher is None:
            raise RuntimeError("DistillStep.multi_step_backward needs the Arc2Face teacher")
        x0, t, noise, face_embs, tokens = batch["x0"], batch["t"], batch["noise"], batch["face_embs"], batch["tokens"]
        img_mask, fg_mask = batch_masks(batch)
        ND = int(num_denoising_steps)
        with torch.no_grad():
            prompt_embs, _ = arc2face_forward_face_embs(self.tokenizer, self.arc2face, face_embs, input_max_length=21,
                                                        return_full_and_core_embs=True)
            ddpm = _QSampleOnly(self._acp(x0.device))
            preds, pred_x0s, noises, ts = self.teacher(ddpm, x0, noise, t, prompt_embs, num_denoising_steps=ND)
        loss_start_step = max(0, ND - 7 // x0.shape[0])
        c = self.context(face_embs, tokens)
        norm = 1.0 / math.sqrt(ND)
        total, grad_c = None, None
        if use_graph:
            g = self.graphed()
        for s in range(loss_start_step, ND):
            x_s = self.q_sample(pred_x0s[s - 1].float(), ts[s], noises[s].float())
            if use_graph:
                ls, gs = g(x_s, ts[s], c.detach(), preds[s].float(), img_mask, fg_mask)
                grad_c = gs if grad_c is None else grad_c + gs
            else:
                eps = unet_forward_train(self.unet, x_s, ts[s], c, self.student_extra_info(img_mask))
                ls = self.recon_loss(eps, preds[s].float(), img_mask, fg_mask)
            total = ls if total is None else total + ls
        total = total * norm
        if use_graph:
            c.backward(grad_c * (norm / accum))
            return total
        (total / accum).backward()
        return total.detach()

    def micro_backward(self, batch: Dict[str, torch.Tensor], accum: int = 1, use_graph: bool = False) -> torch.Tensor:
        """loss / accum backpropagated into the trainable parameters' .grad; returns the detached loss (no host sync).
        use_graph: UNet forward + backward-to-context replayed from one CUDA graph (train.GraphedUNetLoss)."""
        x0, t, noise, face_embs, tokens = batch["x0"], batch["t"], batch["noise"], batch["face_embs"], batch["tokens"]
        img_mask, fg_mask = batch_masks(batch)
        teacher_eps = batch.get("teacher_eps")
        if teacher_eps is None:
            teacher_eps = self.teacher_eps(x0, t, noise, face_embs)
        if not use_graph:
            loss = self.loss(x0, t, noise, teacher_eps, face_embs, tokens, img_mask, fg_mask)
            (loss / accum).backward()
            return loss.detach()
        c = self.context(face_embs, tokens)
        loss, grad_c = self.graphed()(self.q_sample(x0, t, noise), t, c.detach(), teacher_eps, img_mask, fg_mask)
        c.backward(grad_c * (1.0 / accum))
        return loss

    def micro_step(self, batch: Dict[str, torch.Tensor], accum: int = 1) -> float:
        loss = self.loss(batch["x0"], batch["t"], batch["noise"], batch.get("teacher_eps"), batch["face_embs"], batch["tokens"],
                         *batch_masks(batch))
        (loss / accum).backward()
        return float(loss.detach())


class GraphedAccumStep:
    """ALL micro-batches of one optimizer step of DistillStep replayed from one CUDA graph.

    * The conditioning (Arc2Face prompt, SubjBasisGenerator, frozen CLIP) depends on the identities and prompts only,
      not on the UNet: it runs ONCE on the concatenation of the micro-batches (its GEMMs have 77 rows per sample and are
      latency-bound, so 8 samples cost what 4 do), the UNet forward + backward runs per micro-batch on its slice of the
      context, and the conditioning backward runs once on the concatenated context gradients.  The parameter gradients
      are the same sums the per-micro-batch loop accumulates (embedding_manager / ddpm.py:595-633 with
      accumulate_grad_batches), up to fp32 summation order.  With fuse_unet (default) the frozen UNet also runs once,
      on all micro-batches as one batch (same gradient of sum_k MSE_k / accum).
    * Every parameter gradient is accumulated in place into its GradBucket view; nothing on the path reads back to the
      host (no .item(), no nonzero, token ids and the schedule resident on the device), so the only per-replay host
      work is copying the batches into the static buffers.
    Recaptured when the geometry, the set of masks the micro-batches carry (MASK_KEYS: static buffers too), the
    parameter storage (Prodigy re-binds parameters into its bucket at its first step) or a weight pack of a frozen
    module changes."""

    KEYS = ("x0", "t", "noise", "face_embs", "tokens", "teacher_eps")

    def __init__(self, step: "DistillStep", bucket: GradBucket, accum: int, fuse_unet: bool = True):
        self.step, self.bucket, self.accum, self.fuse_unet = step, bucket, accum, fuse_unet
        self._g = {}

    def _keys(self, batch):
        return self.KEYS + tuple(k for k in MASK_KEYS if batch.get(k) is not None)

    def _key(self, batches):
        from .attention import PackedModule
        ps = self.bucket.params
        return (tuple((k, tuple(b[k].shape), b[k].dtype) for b in batches for k in self._keys(b)), ps[0].data_ptr(),
                ps[-1].data_ptr(), PackedModule.PACK_EPOCH, self.fuse_unet)

    def _build(self, batches):
        st = {"in": [{k: b[k].clone() for k in self._keys(b)} for b in batches]}
        step, n = self.step, len(batches)

        def run():
            ins = st["in"]
            c = step.context(torch.cat([i["face_embs"] for i in ins]), torch.cat([i["tokens"] for i in ins]), groups=n)
            rows = c.shape[0] // n                                  # (b l) order: a micro-batch owns a contiguous row range
            losses, grads = [], []
            same = all(i["x0"].shape == ins[0]["x0"].shape for i in ins)
            if self.fuse_unet and same:
                # The frozen UNet sees the micro-batches as ONE batch (the accumulation loop exists for the memory of
                # smaller GPUs; 180 GB hold the activations of all of them, and the kernels fill the SMs better):
                # sum_k MSE_k / accum has the same gradient either way.
                ck = c.detach().clone().requires_grad_(True)
                x0, t, noise = (torch.cat([i[key] for i in ins]) for key in ("x0", "t", "noise"))
                img_mask = torch.cat([i["img_mask"] for i in ins]) if "img_mask" in ins[0] else None
                eps = unet_forward_train(step.unet, step.q_sample(x0, t, noise), t, ck, step.student_extra_info(img_mask))
                per = eps.shape[0] // n
                ls = [step.recon_loss(eps[k * per:(k + 1) * per], i["teacher_eps"], i.get("img_mask"), i.get("fg_mask"))
                      for k, i in enumerate(ins)]
                (g,) = torch.autograd.grad(sum(ls), ck)
                c.backward(g * (1.0 / self.accum))
                return torch.stack([l.detach() for l in ls])
            for k, i in enumerate(ins):
                ck = c.detach()[k * rows:(k + 1) * rows].clone().requires_grad_(True)
                eps = unet_forward_train(step.unet, step.q_sample(i["x0"], i["t"], i["noise"]), i["t"], ck,
                                         step.student_extra_info(i.get("img_mask")))
                loss = step.recon_loss(eps, i["teacher_eps"], i.get("img_mask"), i.get("fg_mask"))
                (g,) = torch.autograd.grad(loss, ck)
                losses.append(loss.detach())
                grads.append(g)
            c.backward(torch.cat(grads) * (1.0 / self.accum))
            return torch.stack(losses)

        for p, v in zip(self.bucket.params, self.bucket.views):
            p.grad = v                                  # AccumulateGrad then adds in place (captured as kernels)
        keep = self.bucket.flat.clone()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):                          # fills the lazy caches (frozen packs, device token ids)
                run()
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            st["losses"] = run()
        self.bucket.flat.copy_(keep)
        st["graph"] = graph
        return st

    def __call__(self, batches: Sequence[Dict[str, torch.Tensor]]) -> torch.Tensor:
        """-> the micro-batch losses [accum] (detached); the gradients of sum_i loss_i / accum are added to the bucket."""
        check_mask_presence(batches)
        for b in batches:
            batch_masks(b)
        key = self._key(batches)
        st = self._g.get(key)
        if st is None:
            self._g.clear()                             # one live geometry: a stale capture holds GBs of activations
            st = self._g[key] = self._build(batches)
        for dst, b in zip(st["in"], batches):
            for k in dst:
                dst[k].copy_(b[k])
        st["graph"].replay()
        return st["losses"].clone()


class Stage1Trainer:
    """One optimizer step of the Stage-1 distillation (training_step ddpm.py:595-633 around guided_denoise :2483-2532):
    `accum` micro-batches -> gradients accumulate in the flat bucket -> one all-reduce (mean over ranks) -> clip by norm
    0.5 -> Prodigy (ldm/prodigy.py) on the same bucket.
    use_graph: "step" (default) - the micro-batches of an optimizer step are ONE CUDA graph with the conditioning
    batched across them (GraphedAccumStep); True - only the frozen UNet's forward + backward-to-context is a graph
    (train.GraphedUNetLoss), the conditioning runs per micro-batch on the eager tape; False - everything eager."""

    def __init__(self, step: "DistillStep", params: Sequence[torch.nn.Parameter], world_size: int = 1, group=None,
                 accum: int = 2, max_grad_norm: float = 0.5, optimizer=None, use_graph="step"):
        from .prodigy import Prodigy
        self.step, self.world_size, self.group = step, world_size, group
        self.accum, self.max_grad_norm = accum, max_grad_norm
        self.bucket = GradBucket(params)
        self.optimizer = optimizer if optimizer is not None else Prodigy(self.bucket.params)
        self.use_graph = use_graph
        self._gstep = GraphedAccumStep(step, self.bucket, accum) if use_graph == "step" else None
        self.allreduce_ms = None

    def optimizer_step(self, batches: Sequence[Dict[str, torch.Tensor]], time_allreduce: bool = False):
        """-> {"loss": 0-d tensor (mean over the micro-batches), "grad_norm": 0-d tensor (before clipping)}."""
        if len(batches) != self.accum:
            raise ValueError(f"expected {self.accum} micro-batches, got {len(batches)}")
        check_mask_presence(batches)
        for b in batches:
            batch_masks(b)
        self.bucket.begin_step()
        if self._gstep is not None:
            # the teacher (no grad) runs outside the captured step
            batches = [b if b.get("teacher_eps") is not None else
                       dict(b, teacher_eps=self.step.teacher_eps(b["x0"], b["t"], b["noise"], b["face_embs"]))
                       for b in batches]
            loss_sum = self._gstep(batches).sum()
        else:
            loss_sum = None
            for b in batches:
                li = self.step.micro_backward(b, accum=self.accum, use_graph=bool(self.use_graph))
                loss_sum = li if loss_sum is None else loss_sum + li
        if time_allreduce and self.world_size > 1:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            self.bucket.allreduce(self.world_size, group=self.group)
            e1.record()
            e1.synchronize()
            self.allreduce_ms = e0.elapsed_time(e1)
        else:
            self.bucket.allreduce(self.world_size, group=self.group)
        gn = self.bucket.clip_(self.max_grad_norm)
        self.optimizer.step(self.bucket.flat)
        return {"loss": loss_sum / self.accum, "grad_norm": gn}
