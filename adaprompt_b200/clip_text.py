"""Host mirror of the CLIP text transformer as the reference drives it (askerlee/adaprompt):

  * adaface/arc2face_models.py: CLIPTextModelWrapper :175 (forward :178-280 - accepts pre-built token embeddings,
    returns a weighted sum of the last hidden states before the final LayerNorm), CLIPAttentionMKV :16-173,
    extend_clip_attention_MKV_multiplier :285-302;
  * ldm/modules/encoders/modules.py: FrozenCLIPEmbedder :179-463 (embeddings_forward :195-223 calls the embedding
    manager on the token embeddings; last-layers skip weighting :361-368).

Same class / attribute names and HuggingFace `state_dict` keys (text_model.encoder.layers.N.self_attn.q_proj.weight,
...), so reference checkpoints load unchanged.  The torch.nn layers only hold parameters; the arithmetic runs in
libadaface_b200.so: LayerNorm -> fused [q|k|v] GEMM (+bias) -> 77-token causal attention (MKV aware) -> out_proj
GEMM (+bias +residual) -> LayerNorm -> fc1 GEMM (+bias, quick_gelu epilogue) -> fc2 GEMM (+bias +residual); fp32
residual stream, bf16 tensor-core operands.  The transformers package is NOT used (the installed 5.5.0 drops the
causal mask inside the reference wrappers - SURVEY.md section 8(c)).
"""
from __future__ import annotations

import types
from typing import Optional, Sequence

import torch
from torch import nn

from . import ops
from .attention import PackedModule


class CLIPTextConfigLite:
    """The openai/clip-vit-large-patch14 text tower (the only configuration the reference uses)."""

    def __init__(self, hidden_size=768, intermediate_size=3072, num_attention_heads=12, num_hidden_layers=12,
                 vocab_size=49408, max_position_embeddings=77, layer_norm_eps=1e-5, hidden_act="quick_gelu",
                 attention_dropout=0.0, eos_token_id=2):
        if hidden_act != "quick_gelu" or hidden_size // num_attention_heads != 64:
            raise NotImplementedError("only quick_gelu and head_dim 64 (CLIP-L/14 text) are implemented")
        self.hidden_size, self.intermediate_size = hidden_size, intermediate_size
        self.num_attention_heads, self.num_hidden_layers = num_attention_heads, num_hidden_layers
        self.vocab_size, self.max_position_embeddings = vocab_size, max_position_embeddings
        self.layer_norm_eps, self.hidden_act, self.attention_dropout = layer_norm_eps, hidden_act, attention_dropout
        self.eos_token_id = eos_token_id
        self.use_return_dict = True
        self.output_attentions = False
        self.output_hidden_states = False


class CLIPAttentionMKV(nn.Module):
    """arc2face_models.py:16-173: multi-head attention whose k / v projections emit `multiplier` keys / values per
    token.  multiplier = 1 is the stock HF CLIPAttention."""

    def __init__(self, config, multiplier=2):
        super().__init__()
        self.config = config
        self.embed_dim = config.hidden_size
        self.num_heads = config.num_attention_heads
        self.head_dim = self.embed_dim // self.num_heads
        self.scale = self.head_dim ** -0.5
        self.dropout = config.attention_dropout
        self.multiplier = multiplier
        self.k_proj = nn.Linear(self.embed_dim, self.embed_dim * multiplier)
        self.v_proj = nn.Linear(self.embed_dim, self.embed_dim * multiplier)
        self.q_proj = nn.Linear(self.embed_dim, self.embed_dim)
        self.out_proj = nn.Linear(self.embed_dim, self.embed_dim)

    def extend_weights(self, clip_attn_layer, layer_idx, multiplier, noise_std=0.1, noise_std_is_relative=True,
                       keep_norm=False, verbose=False):
        """arc2face_models.py:46-85: repeat the k / v projections `multiplier` times, noise on the extra copies."""
        self.multiplier *= multiplier
        E = self.embed_dim
        with torch.no_grad():
            for n in ("q_proj", "out_proj"):
                getattr(self, n).weight.data = getattr(clip_attn_layer, n).weight.data.clone()
                getattr(self, n).bias.data = getattr(clip_attn_layer, n).bias.data.clone()
            for n in ("v_proj", "k_proj"):
                src = getattr(clip_attn_layer, n)
                lin = nn.Linear(E, src.weight.shape[0] * multiplier).to(src.weight.device)
                lin.bias.data = src.bias.data.repeat(multiplier)
                lin.weight.data = src.weight.data.repeat(multiplier, 1)
                if noise_std > 0:
                    d0 = src.weight.shape[0]
                    extra = lin.weight.data[d0:]
                    std = extra.std() * noise_std if noise_std_is_relative else noise_std
                    noised = extra + torch.randn_like(extra) * std
                    if keep_norm:
                        noised = noised * (extra.norm() / noised.norm())
                    lin.weight.data[d0:] = noised
                setattr(self, n, lin)


CLIPAttention = CLIPAttentionMKV  # multiplier 1


class CLIPMLP(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.fc1 = nn.Linear(config.hidden_size, config.intermediate_size)
        self.fc2 = nn.Linear(config.intermediate_size, config.hidden_size)


class CLIPEncoderLayer(PackedModule):
    def __init__(self, config):
        super().__init__()
        self.embed_dim = config.hidden_size
        self.self_attn = CLIPAttentionMKV(config, 1)
        self.layer_norm1 = nn.LayerNorm(self.embed_dim, eps=config.layer_norm_eps)
        self.mlp = CLIPMLP(config)
        self.layer_norm2 = nn.LayerNorm(self.embed_dim, eps=config.layer_norm_eps)

    def _pack(self):
        a = self.self_attn
        E, H, hd, m = a.embed_dim, a.num_heads, a.head_dim, a.k_proj.weight.shape[0] // a.embed_dim
        f = lambda t: t.detach().float().contiguous()

        def kv_rows(w):
            # reference key order (arc2face_models.py:117-131): key r of token t = columns [r*E, (r+1)*E), head h at
            # r*E + h*hd  ->  kernel order [head][r][hd]
            return w.reshape(m, H, hd, *w.shape[1:]).transpose(0, 1).reshape(m * E, *w.shape[1:])

        wqkv = torch.cat([f(a.q_proj.weight), kv_rows(f(a.k_proj.weight)), kv_rows(f(a.v_proj.weight))], 0)
        bqkv = torch.cat([f(a.q_proj.bias), kv_rows(f(a.k_proj.bias)), kv_rows(f(a.v_proj.bias))], 0)
        return {"m": m, "wqkv": wqkv.to(torch.bfloat16).contiguous(), "bqkv": bqkv.contiguous(),
                "wo": a.out_proj.weight.detach().to(torch.bfloat16).contiguous(), "bo": f(a.out_proj.bias),
                "w1": self.mlp.fc1.weight.detach().to(torch.bfloat16).contiguous(), "b1": f(self.mlp.fc1.bias),
                "w2": self.mlp.fc2.weight.detach().to(torch.bfloat16).contiguous(), "b2": f(self.mlp.fc2.bias),
                "ln1": (f(self.layer_norm1.weight), f(self.layer_norm1.bias), float(self.layer_norm1.eps)),
                "ln2": (f(self.layer_norm2.weight), f(self.layer_norm2.bias), float(self.layer_norm2.eps))}

    def invalidate_packed(self):
        super().invalidate_packed()

    def _run(self, h: torch.Tensor, B: int, L: int, causal: bool = True) -> torch.Tensor:
        """h fp32 [B*L, E] -> fp32 [B*L, E]."""
        pk = self.packed()
        a = self.self_attn
        E, H, m = a.embed_dim, a.num_heads, pk["m"]
        T, dev = h.shape[0], h.device
        x = torch.empty(T, E, dtype=torch.bfloat16, device=dev)
        ops.layernorm(h, pk["ln1"][0], pk["ln1"][1], pk["ln1"][2], x)
        qkv = torch.empty(T, E * (1 + 2 * m), dtype=torch.bfloat16, device=dev)
        ops.gemm(x, pk["wqkv"], qkv, bias=pk["bqkv"])
        o = torch.empty(T, E, dtype=torch.bfloat16, device=dev)
        ops.attention_small(qkv, o, B=B, heads=H, L=L, k_off=E, v_off=E + E * m, mult=m, scale=a.scale, causal=causal)
        h1 = torch.empty(T, E, dtype=torch.float32, device=dev)
        ops.gemm(o, pk["wo"], h1, bias=pk["bo"], residual=h)
        ops.layernorm(h1, pk["ln2"][0], pk["ln2"][1], pk["ln2"][2], x)
        u = torch.empty(T, pk["w1"].shape[0], dtype=torch.bfloat16, device=dev)
        ops.gemm(x, pk["w1"], u, bias=pk["b1"], act=1)
        h2 = torch.empty(T, E, dtype=torch.float32, device=dev)
        ops.gemm(u, pk["w2"], h2, bias=pk["b2"], residual=h1)
        return h2


class CLIPEncoder(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.layers = nn.ModuleList([CLIPEncoderLayer(config) for _ in range(config.num_hidden_layers)])


class CLIPTextEmbeddings(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.token_embedding = nn.Embedding(config.vocab_size, config.hidden_size)
        self.position_embedding = nn.Embedding(config.max_position_embeddings, config.hidden_size)
        self.register_buffer("position_ids", torch.arange(config.max_position_embeddings).expand((1, -1)),
                             persistent=False)

    def forward(self, input_ids=None, position_ids=None, inputs_embeds=None, embedding_manager=None):
        """CLIPTextEmbeddings.forward as patched at modules.py:195-223: token lookup -> [embedding manager] -> + pos."""
        if position_ids is not None:
            raise NotImplementedError("explicit position_ids")
        tw = self.token_embedding.weight
        if not tw.is_cuda:
            raise RuntimeError("CLIPTextEmbeddings: parameters must be on a CUDA device (no CPU fallback)")
        if inputs_embeds is None:
            inputs_embeds = ops.gather_rows(tw.detach().float().contiguous(), input_ids.contiguous())
        else:
            inputs_embeds = inputs_embeds.detach().float().clone()
        if embedding_manager is not None:
            inputs_embeds = embedding_manager(input_ids, inputs_embeds)
        inputs_embeds = inputs_embeds.contiguous()
        return ops.add_pos(inputs_embeds, self.position_embedding.weight.detach().float().contiguous())


class CLIPTextTransformer(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.config = config
        self.embeddings = CLIPTextEmbeddings(config)
        self.encoder = CLIPEncoder(config)
        self.final_layer_norm = nn.LayerNorm(config.hidden_size, eps=config.layer_norm_eps)
        self.eos_token_id = config.eos_token_id
        self.last_layers_skip_weights = None   # set by FrozenCLIPEmbedder.set_last_layers_skip_weights

    def encode(self, h: torch.Tensor, layer_weights: Optional[Sequence[float]]) -> torch.Tensor:
        """h fp32 [B, L, E] (embeddings incl. positions) -> final-LayerNormed fp32 [B, L, E].  layer_weights:
        already-normalised weights of the last len(w) hidden states, or None for the last state only."""
        B, L, E = h.shape
        x = h.reshape(B * L, E)
        n_keep = len(layer_weights) if layer_weights is not None else 1
        states = [x]
        for layer in self.encoder.layers:
            x = layer._run(x, B, L)
            states.append(x)
            if len(states) > n_keep:
                states.pop(0)
        if layer_weights is not None:
            w = [float(v) for v in layer_weights]
            if len(w) == 1:
                mixed = states[-1]
            elif len(w) in (2, 3):
                mixed = ops.weighted_sum(states[0], states[1], states[2] if len(w) == 3 else None, w)
            else:
                raise NotImplementedError("more than 3 weighted hidden states")
        else:
            mixed = states[-1]
        out = torch.empty(B * L, E, dtype=torch.float32, device=h.device)
        ln = self.final_layer_norm
        ops.layernorm(mixed, ln.weight.detach().float().contiguous(), ln.bias.detach().float().contiguous(), float(ln.eps), out)
        return out.reshape(B, L, E)


class CLIPTextModelWrapper(nn.Module):
    """arc2face_models.py:175-302."""

    def __init__(self, config: Optional[CLIPTextConfigLite] = None):
        super().__init__()
        self.config = config or CLIPTextConfigLite()
        self.text_model = CLIPTextTransformer(self.config)

    @property
    def dtype(self):
        return self.text_model.final_layer_norm.weight.dtype

    @property
    def device(self):
        return self.text_model.final_layer_norm.weight.device

    def forward(self, input_ids=None, attention_mask=None, position_ids=None, output_attentions=None,
                output_hidden_states=None, return_dict=None, input_token_embs=None,
                hidden_state_layer_weights=None, return_token_embs=False):
        tm = self.text_model
        if input_ids is None:
            raise ValueError("You have to specify input_ids")
        input_ids = input_ids.view(-1, input_ids.shape[-1])
        if return_token_embs:                                                                       # :191-192
            return ops.gather_rows(tm.embeddings.token_embedding.weight.detach().float().contiguous(),
                                   input_ids.contiguous())
        if attention_mask is not None or output_attentions:
            raise NotImplementedError("attention_mask / output_attentions are not used on the AdaFace path")
        h = tm.embeddings(input_ids=input_ids, position_ids=position_ids, inputs_embeds=input_token_embs)  # :210
        w = None
        if hidden_state_layer_weights is not None:                                                  # :236-246
            hw = hidden_state_layer_weights.detach().float()
            if hw.dim() == 2 and hw.shape[1] != 1:
                raise NotImplementedError("per-channel hidden_state_layer_weights")
            hw = hw.reshape(-1)
            w = (hw / hw.sum()).tolist()
        last = tm.encode(h, w)                                                                      # :220,:248
        eos = input_ids.to(torch.int).argmax(dim=-1) if tm.eos_token_id == 2 else \
            (input_ids.to(torch.int) == tm.eos_token_id).int().argmax(dim=-1)
        pooled = last[torch.arange(last.shape[0], device=last.device), eos]
        if return_dict is False:
            return (last, pooled)
        return _Output(last_hidden_state=last, pooler_output=pooled, hidden_states=None, attentions=None)

    def extend_clip_attention_MKV_multiplier(self, begin_layer_idx=-1, end_layer_idx=-1, multiplier=2, noise_std=0.1):
        """arc2face_models.py:285-302.  Multipliers compound across calls.  The forward runs any total multiplier up to 4,
        but the training backward (attention_small_bwd_kernel) holds the scores of a 77-token layer in shared memory and
        refuses a total above 2 with ValueError."""
        n = 0
        for layer_idx, layer in enumerate(self.text_model.encoder.layers):
            if begin_layer_idx >= 0 and layer_idx < begin_layer_idx:
                continue
            if end_layer_idx >= 0 and layer_idx >= end_layer_idx:
                break
            old = layer.self_attn
            new = CLIPAttentionMKV(old.config, old.multiplier)
            new.k_proj, new.v_proj = old.k_proj, old.v_proj
            new.extend_weights(old, layer_idx, multiplier, noise_std, verbose=True)
            layer.self_attn = new
            layer.invalidate_packed()
            n += 1
        return n


class _Output(tuple):
    """BaseModelOutputWithPooling stand-in: indexable like the HF tuple, with the same attribute names."""

    def __new__(cls, last_hidden_state, pooler_output, hidden_states=None, attentions=None):
        o = super().__new__(cls, (last_hidden_state, pooler_output))
        o.last_hidden_state, o.pooler_output = last_hidden_state, pooler_output
        o.hidden_states, o.attentions = hidden_states, attentions
        return o


class _CLIPTextModelHolder(nn.Module):
    """`FrozenCLIPEmbedder.transformer` (a CLIPTextModel): holds `text_model` so that SD checkpoints' keys
    `cond_stage_model.transformer.text_model.*` load unchanged."""

    def __init__(self, config):
        super().__init__()
        self.config = config
        self.text_model = CLIPTextTransformer(config)


class FrozenCLIPEmbedder(nn.Module):
    """ldm/modules/encoders/modules.py:179-463.  `tokenizer` is any callable with the CLIPTokenizer call protocol
    (there are no vocabulary files offline); token tensors can be passed instead of strings."""

    def __init__(self, version="openai/clip-vit-large-patch14", device="cuda", max_length=77,
                 last_layers_skip_weights=(0.5, 0.5), randomize_clip_skip_weights=False, tokenizer=None, config=None):
        super().__init__()
        if randomize_clip_skip_weights:
            raise NotImplementedError("randomize_clip_skip_weights (training-time Dirichlet sampling)")
        self.tokenizer = tokenizer
        self.transformer = _CLIPTextModelHolder(config or CLIPTextConfigLite())
        self.device = device
        self.max_length = max_length
        self.set_last_layers_skip_weights(last_layers_skip_weights)
        self.dedup_layer_copies = True
        for p in self.parameters():
            p.requires_grad = False

    def set_last_layers_skip_weights(self, weights, use_as_dirichlet_weights=False):
        """modules.py:405-420: normalised to sum 1; the LAST element weighs the last layer."""
        if use_as_dirichlet_weights:
            raise NotImplementedError("Dirichlet skip weights")
        s = float(sum(weights))
        self.transformer.text_model.last_layers_skip_weights = [float(w) / s for w in weights]

    def tokenize(self, text):
        if torch.is_tensor(text):
            return text
        if self.tokenizer is None:
            raise RuntimeError("FrozenCLIPEmbedder: no tokenizer set (CLIP vocabulary files are not available offline); "
                               "pass token ids or supply `tokenizer`")
        enc = self.tokenizer(text, truncation=True, max_length=self.max_length, return_length=True,
                             return_overflowing_tokens=False, padding="max_length", return_tensors="pt")
        return enc["input_ids"] if isinstance(enc, dict) else enc.input_ids

    def forward(self, text, embedding_manager=None, **kwargs):
        tm = self.transformer.text_model
        dev = tm.final_layer_norm.weight.device
        tokens = self.tokenize(text).to(dev)
        tw = tm.embeddings.token_embedding.weight.detach().float().contiguous()
        emb = ops.gather_rows(tw, tokens.contiguous())                                             # :207-208
        identical = False
        if embedding_manager is not None:
            emb = embedding_manager(tokens, emb)                                                    # :212-213
            identical = bool(getattr(embedding_manager, "layer_copies_identical", False))
        B = tokens.shape[0]
        rep = emb.shape[0] // B
        pos = tm.embeddings.position_embedding.weight.detach().float().contiguous()
        if rep > 1 and identical and self.dedup_layer_copies:
            # SURVEY.md section 8(f) N2: the 16 layer copies of a sequence are bit-identical when no background token
            # is present (SubjBasisGenerator repeats the same core embeddings, subj_basis_generator.py:558), so one
            # copy is encoded and broadcast - bit-identical to encoding all 16.
            one = emb.reshape(B, rep, *emb.shape[1:])[:, 0].contiguous()
            z = tm.encode(ops.add_pos(one, pos), tm.last_layers_skip_weights)
            return z.unsqueeze(1).expand(B, rep, *z.shape[1:]).reshape(B * rep, *z.shape[1:]).contiguous()
        return tm.encode(ops.add_pos(emb.contiguous(), pos), tm.last_layers_skip_weights)           # :260-283,:361-370

    def encode(self, text, **kwargs):
        return self(text, **kwargs)
