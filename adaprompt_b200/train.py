"""Stage-1 distillation step on the B200 C ABI (SURVEY.md section 8 row T1).

Reference: LatentDiffusion.guided_denoise (ldm/models/diffusion/ddpm.py:2483-2532) runs UNetModel.forward WITH grad;
the UNet weights are frozen (ddpm.py:783-786), so its backward is activation gradients only - they flow to the
trainable SubjBasisGenerator through the 16 layerwise cross-attention contexts (openaimodel.py:866,978).  The loss is
the (masked) MSE against the teacher's noise prediction (calc_recon_loss ddpm.py:3571-3595, :3010-3037): distill_loss
without image masks, calc_recon_loss with them.  A batch of real face images carries an image mask (which latent pixels
hold image rather than augmentation padding), used by the student UNet as a self-attention key mask, and a face mask;
both weight the loss.

torch.autograd is used as the *tape* only (plumbing: which op ran, which buffers it saved); every forward and
backward op below is a hand-written kernel behind the C ABI:
  * dgrad GEMMs / convolutions = the forward tcgen05 kernels on transposed / flipped weight packs;
  * GroupNorm(+SiLU), LayerNorm, GEGLU backward = train.cu;
  * attention backward = five batched strided contractions per (sample, head) with the softmax recomputed from the
    forward kernel's log-sum-exp in the GEMM epilogue (bgemm.cu; materialised P - a fused tcgen05 backward is the
    next step, see DESIGN.md);
  * weight gradients (trainable CLIP text layers of SubjBasisGenerator.prompt2token_proj) = tensor-core GEMMs over
    transposed operands.
Layout as in the inference path: NHWC / tokens x channels, fp32 residual stream, bf16 GEMM operands.
"""
from __future__ import annotations

import math
from typing import Optional

import torch
from torch.autograd import Function

from . import ops
from .attention import BasicTransformerBlock, CrossAttention, FeedForward, SpatialTransformer
from .packing import head_pad, pack_conv3x3
from .unet import L2CA, ConvIn, Downsample, ResBlock, TimestepEmbedSequential, UNetModel, Upsample

LN2 = math.log(2.0)


def _t(w: torch.Tensor) -> torch.Tensor:
    return w.t().contiguous()


def _flip_conv_pack(w_oihw: torch.Tensor) -> torch.Tensor:
    """Weight pack of the conv that computes the input gradient of a 3x3 / pad 1 conv: channels swapped, taps flipped."""
    return pack_conv3x3(w_oihw.detach().permute(1, 0, 2, 3).flip(2, 3).contiguous())


def bwd_packs(m) -> dict:
    """Lazily built transposed weight packs of one host-mirror module (dgrad operands)."""
    pb = m.__dict__.get("_pk_bwd")
    if pb is not None:
        return pb
    pk = m.packed()
    with torch.no_grad():
        if isinstance(m, ResBlock):
            pb = {"w1": _flip_conv_pack(m.in_layers[2].weight), "w2": _flip_conv_pack(m.out_layers[3].weight)}
            if "ws" in pk:
                pb["ws"] = _t(pk["ws"])
        elif isinstance(m, Upsample):
            pb = {"w": _flip_conv_pack(m.conv.weight)}
        elif isinstance(m, Downsample):
            pb = {"w": _flip_conv_pack(m.op.weight)}
        elif isinstance(m, CrossAttention):
            pb = {k: _t(pk[k]) for k in ("wo", "wv", "wq", "wk") if k in pk}
            if "wqk" in pk:
                pb["wqk"] = _t(pk["wqk"])
        elif isinstance(m, FeedForward):
            w1 = m.net[0].proj.weight.detach().to(torch.bfloat16).contiguous()       # reference row order: value | gate
            pb = {"w1_plain": w1, "b1_plain": m.net[0].proj.bias.detach().float().contiguous(), "w1": _t(w1),
                  "w2": _t(pk["w2"])}
        elif isinstance(m, SpatialTransformer):
            pb = {"w_in": _t(pk["w_in"]), "w_out": _t(pk["w_out"])}
        else:
            raise TypeError(type(m))
    m.__dict__["_pk_bwd"] = pb
    return pb


def _bf16(t: torch.Tensor) -> torch.Tensor:
    if t.dtype == torch.bfloat16:
        return t.contiguous()
    return ops.cast_bf16(t.float().contiguous())


# ------------------------------------------------------------------------------------------------ Functions
class CastBF16(Function):
    @staticmethod
    def forward(ctx, x):
        return ops.cast_bf16(x.contiguous())

    @staticmethod
    def backward(ctx, dy):
        return dy.float()


class LinearFn(Function):
    """out = x @ W^T + b (+ residual).  x bf16 [T, K]; w bf16 [N, K] pack, wt bf16 [K, N] pack.
    w_param / b_param: the fp32 nn.Parameters when they are trainable (weight gradients), else None."""

    @staticmethod
    def forward(ctx, x, w, wt, bias, residual, out_dtype, w_param, b_param, act):
        T = x.shape[0]
        out = torch.empty(T, w.shape[0], dtype=out_dtype, device=x.device)
        if act:  # quick_gelu is applied by a separate Function in training form
            raise NotImplementedError
        ops.gemm(x, w, out, bias=bias, residual=residual)
        ctx.wt = wt
        ctx.has_res = residual is not None
        ctx.x_dtype = x.dtype
        ctx.save_for_backward(x if ctx.needs_input_grad[6] else None)
        ctx.K = x.shape[1]
        return out

    @staticmethod
    def backward(ctx, dout):
        (x,) = ctx.saved_tensors
        dob = _bf16(dout)
        dx = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty(dob.shape[0], ctx.K, dtype=torch.bfloat16, device=dout.device)
            ops.gemm(dob, ctx.wt, dx)
        dres = dout if (ctx.has_res and ctx.needs_input_grad[4]) else None
        dw = db = None
        if ctx.needs_input_grad[6] and x is not None:
            # dW [N, K] = dY^T [N, T] . X [T, K]: both operands transposed so that T is the contraction (K-major) dim
            doT = ops.transpose_to_bf16(dob)
            xT = ops.transpose_to_bf16(x)
            dw = torch.empty(doT.shape[0], xT.shape[0], dtype=torch.float32, device=dout.device)
            ops.gemm(doT, xT, dw)
        if ctx.needs_input_grad[7]:
            db = dout.float().sum(0)
        return dx, None, None, None, dres, None, dw, db, None


def linear(x, w, wt, bias=None, residual=None, out_dtype=torch.float32, w_param=None, b_param=None):
    return LinearFn.apply(x, w, wt, bias, residual, out_dtype, w_param, b_param, 0)


class GroupNormFn(Function):
    """GroupNorm(32) [+SiLU]: x fp32 NHWC -> bf16 (util.py:217-219, attention.py:71-72)."""

    @staticmethod
    def forward(ctx, x, gamma, beta, eps, silu):
        x = x.contiguous()
        mr = ops.groupnorm_mean_rstd(x, ops.groupnorm_stats(x), eps)
        y = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
        ops.groupnorm_apply_mr(x, mr, gamma, beta, silu, y)
        ctx.save_for_backward(x, mr, gamma, beta)
        ctx.silu = silu
        return y

    @staticmethod
    def backward(ctx, dy):
        x, mr, gamma, beta = ctx.saved_tensors
        return ops.groupnorm_bwd(x, mr, gamma, beta, ctx.silu, dy.contiguous()), None, None, None, None


class LayerNormFn(Function):
    """nn.LayerNorm: x fp32 [T, C] -> bf16 | fp32.  gamma / beta may be trainable parameters (CLIP text layers)."""

    @staticmethod
    def forward(ctx, x, gamma, beta, eps, out_dtype):
        x = x.contiguous()
        y = torch.empty(x.shape, dtype=out_dtype, device=x.device)
        g, b = gamma.detach().float().contiguous(), beta.detach().float().contiguous()
        ops.layernorm(x, g, b, eps, y)
        ctx.save_for_backward(x, g)
        ctx.eps = eps
        return y

    @staticmethod
    def backward(ctx, dy):
        x, g = ctx.saved_tensors
        dg = db = None
        if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
            dg = torch.zeros_like(g)
            db = torch.zeros_like(g)
        dx = ops.layernorm_bwd(x, g, ctx.eps, dy.contiguous(), None, dg, db)
        return dx, dg, db, None, None


class Conv3x3Fn(Function):
    """3x3 / pad 1 / stride 1 conv on bf16 NHWC (+bias +per-sample row bias +fp32 residual) -> fp32."""

    @staticmethod
    def forward(ctx, y, w, w_bwd, bias, rowbias, residual):
        B, H, W, _ = y.shape
        out = torch.empty(B, H, W, w.shape[0], dtype=torch.float32, device=y.device)
        ops.conv3x3(y, w, out, bias=bias, rowbias=rowbias, residual=residual)
        ctx.w_bwd = w_bwd
        ctx.has_res = residual is not None
        return out

    @staticmethod
    def backward(ctx, dout):
        dout = dout.contiguous()
        B, H, W, _ = dout.shape
        dy = torch.empty(B, H, W, ctx.w_bwd.shape[0], dtype=torch.bfloat16, device=dout.device)
        ops.conv3x3(ops.cast_bf16(dout), ctx.w_bwd, dy)
        return dy, None, None, None, None, (dout if ctx.has_res else None)


class UpsampleConvFn(Function):
    """openaimodel.py:95-123: nearest x2 + conv3x3; backward = dgrad conv + 2x2 sum-pool."""

    @staticmethod
    def forward(ctx, x, w, w_bwd, bias):
        x = x.contiguous()
        B, H, W, C = x.shape
        up = torch.empty(B, 2 * H, 2 * W, C, dtype=torch.bfloat16, device=x.device)
        ops.upsample2x_cast(x, up)
        out = torch.empty(B, 2 * H, 2 * W, w.shape[0], dtype=torch.float32, device=x.device)
        ops.conv3x3(up, w, out, bias=bias)
        ctx.w_bwd = w_bwd
        return out

    @staticmethod
    def backward(ctx, dout):
        dout = dout.contiguous()
        B, H2, W2, _ = dout.shape
        dup = torch.empty(B, H2, W2, ctx.w_bwd.shape[0], dtype=torch.float32, device=dout.device)
        ops.conv3x3(ops.cast_bf16(dout), ctx.w_bwd, dup)
        return ops.sumpool2x2(dup), None, None, None


class DownsampleConvFn(Function):
    """openaimodel.py:138-164: conv3x3 stride 2; backward = stride-1 dgrad conv over the zero-inserted gradient."""

    @staticmethod
    def forward(ctx, x, w, w_bwd, bias):
        x = x.contiguous()
        B, H, W, C = x.shape
        out = torch.empty(B, H // 2, W // 2, w.shape[0], dtype=torch.float32, device=x.device)
        ops.conv3x3(ops.cast_bf16(x), w, out, stride=2, bias=bias)
        ctx.w_bwd = w_bwd
        return out

    @staticmethod
    def backward(ctx, dout):
        dz = ops.zero_insert2x(dout.contiguous())
        B, H, W, _ = dz.shape
        dx = torch.empty(B, H, W, ctx.w_bwd.shape[0], dtype=torch.float32, device=dout.device)
        ops.conv3x3(dz, ctx.w_bwd, dx)
        return dx, None, None, None


class ConvOutFn(Function):
    """UNetModel.out[2] (openaimodel.py:696): bf16 NHWC [B,H,W,320] -> fp32 NCHW [B,4,H,W]."""

    @staticmethod
    def forward(ctx, y, w_pack8, bias8, w_f32, out_channels):
        B, H, W, C = y.shape
        o8 = torch.empty(B, H, W, w_pack8.shape[0], dtype=torch.float32, device=y.device)
        ops.conv3x3(y, w_pack8, o8, bias=bias8, bn=64)
        out = torch.empty(B, out_channels, H, W, dtype=torch.float32, device=y.device)
        ops.nhwc_to_nchw(o8, out)
        ctx.w_f32, ctx.C = w_f32, C
        return out

    @staticmethod
    def backward(ctx, dout):
        return ops.conv_out_dgrad(dout.contiguous().float(), ctx.w_f32, ctx.C), None, None, None, None


class GegluFn(Function):
    @staticmethod
    def forward(ctx, proj):
        ctx.save_for_backward(proj)
        return ops.geglu_fwd(proj)

    @staticmethod
    def backward(ctx, dh):
        (proj,) = ctx.saved_tensors
        return ops.geglu_bwd(proj, dh.contiguous())


class AttentionFn(Function):
    """softmax(q k^T) v per (sample, head) (attention.py:198-242).  q bf16 [B*Nq, >= h*dp] (pre-scaled, log2 domain),
    k bf16 [B*nk_pad, >= h*dp], v bf16 [B*nk_pad, h*d]; q / k may be column views of one fused [Q|K] buffer.
    Returns o bf16 [B*Nq, h*d].  nk <= nk_pad valid keys per sample.  key_mask: None or uint8 [B, nk] (1 = attend), the
    self-attention key mask of attention.py:223-232; its backward runs the masked kernels."""

    @staticmethod
    def forward(ctx, q, k, v, B, heads, d, Nq, nk, nk_pad, key_mask=None):
        dp = head_pad(d)
        C = heads * d
        dev = q.device
        ldvt = max(64, (B * nk_pad + 7) // 8 * 8)
        vt = ops.transpose_to_bf16(v.contiguous(), ldvt)                     # V^T [C, ldvt] (forward kernel operand)
        o = torch.empty(B * Nq, C, dtype=torch.bfloat16, device=dev)
        lse = torch.empty(B, heads, Nq, dtype=torch.float32, device=dev)
        if key_mask is not None:
            ops.check_key_mask(key_mask, B, nk)
        ops.attention_lse(q, k, vt, o, lse, B=B, heads=heads, Nq=Nq, Nk=nk, d=d, ldq=int(q.stride(0)),
                          ldk=int(k.stride(0)), ldvt=ldvt, kv_stride=nk_pad, key_mask=key_mask)
        ctx.save_for_backward(q, k, v, o, lse)
        ctx.key_mask = key_mask
        ctx.geom = (B, heads, d, dp, Nq, nk, nk_pad)
        return o

    @staticmethod
    def backward(ctx, dO):
        q, k, v, o, lse = ctx.saved_tensors
        B, h, d, dp, Nq, nk, nkp = ctx.geom
        C = h * d
        dev = q.device
        dO = dO.contiguous()
        ldq, ldk = int(q.stride(0)), int(k.stride(0))
        delta = ops.rowdot_heads(dO, o, B, Nq, h, d)                                  # [B, h, Nq]
        km = ctx.key_mask                       # None: the unmasked kernels; else their masked instantiations
        Tq, Tk = B * Nq, B * nkp
        if d in (40, 80) and Nq == nk == nkp and Nq % 128 == 0 and ops.attention_bwd is not None:
            # long self-attention: fused tcgen05 backward (attention_bwd.cu), P / dS never leave the SM
            pad = (lambda t: torch.nn.functional.pad(t.view(-1, h, d), (0, dp - d)).view(-1, h * dp)) if dp != d else (lambda t: t)
            vp, dop = pad(v), pad(dO)
            qT = ops.transpose_to_bf16(q[:, :h * dp].contiguous())
            kT = ops.transpose_to_bf16(k[:, :h * dp].contiguous())
            dOT = ops.transpose_to_bf16(dop)
            dq, dk, dv = ops.attention_bwd(q, k, vp, dop, qT, kT, dOT, lse, delta, B=B, heads=h, N=Nq, d=d, key_mask=km)
            if q.shape[1] != h * dp:
                full = torch.zeros(q.shape, dtype=torch.bfloat16, device=dev)
                full[:, :h * dp] = dq
                dq = full
            if k.shape[1] != h * dp:
                full = torch.zeros(k.shape, dtype=torch.bfloat16, device=dev)
                full[:, :h * dp] = dk
                dk = full
            return dq, dk, dv, None, None, None, None, None, None, None
        qT = ops.transpose_to_bf16(q[:, :h * dp].contiguous())                       # [h*dp, Tq_p]
        kT = ops.transpose_to_bf16(k[:, :h * dp].contiguous())                       # [h*dp, Tk_p]
        dOT = ops.transpose_to_bf16(dO)                                              # [C, Tq_p]
        ldqT, ldkT = qT.shape[1], kT.shape[1]
        P = torch.empty(B, h, Nq, nkp, dtype=torch.bfloat16, device=dev)
        Pt = torch.empty(B, h, nkp, Nq, dtype=torch.bfloat16, device=dev)
        sP = (h * Nq * nkp, Nq * nkp)
        qa, ka = q, k                                                                # views: data_ptr() carries the offset
        # P = exp2(S - lse), P^T likewise (S^T recomputed; padded keys -> 0)
        ops.bgemm(qa, ldq, (Nq * ldq, dp), ka, ldk, (nkp * ldk, dp), P, nkp, sP, M=Nq, N=nkp, K=dp, nb0=B, nb1=h,
                  mode=1, vec=lse, sV=(h * Nq, Nq), valid_cols=nk, key_mask=km)
        ops.bgemm(ka, ldk, (nkp * ldk, dp), qa, ldq, (Nq * ldq, dp), Pt, Nq, sP, M=nkp, N=Nq, K=dp, nb0=B, nb1=h,
                  mode=2, vec=lse, sV=(h * Nq, Nq), valid_rows=nk, key_mask=km)
        # dS = ln2 * P o (dO V^T - delta)  and its transpose
        dS = torch.empty_like(P)
        dSt = torch.empty_like(Pt)
        ops.bgemm(dO, C, (Nq * C, d), v, C, (nkp * C, d), dS, nkp, sP, M=Nq, N=nkp, K=d, nb0=B, nb1=h, mode=3,
                  vec=delta, sV=(h * Nq, Nq), P=P, ldp=nkp, sP=sP, valid_cols=nk, alpha=LN2, key_mask=km)
        ops.bgemm(v, C, (nkp * C, d), dO, C, (Nq * C, d), dSt, Nq, sP, M=nkp, N=Nq, K=d, nb0=B, nb1=h, mode=4,
                  vec=delta, sV=(h * Nq, Nq), P=Pt, ldp=Nq, sP=sP, valid_rows=nk, alpha=LN2, key_mask=km)
        # dQ = dS K, dK = dS^T Q, dV = P^T dO
        dq = torch.zeros(Tq, h * dp, dtype=torch.bfloat16, device=dev)
        dk = torch.zeros(Tk, h * dp, dtype=torch.bfloat16, device=dev)
        dv = torch.zeros(Tk, C, dtype=torch.bfloat16, device=dev)
        ops.bgemm(dS, nkp, sP, kT, ldkT, (nkp, dp * ldkT), dq, h * dp, (Nq * h * dp, dp), M=Nq, N=dp, K=nkp, nb0=B, nb1=h)
        ops.bgemm(dSt, Nq, sP, qT, ldqT, (Nq, dp * ldqT), dk, h * dp, (nkp * h * dp, dp), M=nkp, N=dp, K=Nq, nb0=B, nb1=h)
        ops.bgemm(Pt, Nq, sP, dOT, dOT.shape[1], (Nq, d * dOT.shape[1]), dv, C, (nkp * C, d), M=nkp, N=d, K=Nq, nb0=B,
                  nb1=h)
        # q / k may be views of a wider buffer: return gradients with the views' shapes
        if q.shape[1] != h * dp:
            full = torch.zeros(q.shape, dtype=torch.bfloat16, device=dev)
            full[:, :h * dp] = dq
            dq = full
        if k.shape[1] != h * dp:
            full = torch.zeros(k.shape, dtype=torch.bfloat16, device=dev)
            full[:, :h * dp] = dk
            dk = full
        return dq, dk, dv, None, None, None, None, None, None, None


# ------------------------------------------------------------------------------------------------ modules
def _gn(x, w, b, eps, silu):
    return GroupNormFn.apply(x, w, b, eps, silu)


def resblock_train(rb: ResBlock, x: torch.Tensor, emb_rows: torch.Tensor) -> torch.Tensor:
    """ResBlock._forward (openaimodel.py:259-279) with grad; x fp32 NHWC (already concatenated)."""
    pk, pb = rb.packed(), bwd_packs(rb)
    B, H, W, Cin = x.shape
    y = _gn(x, pk["gn1_w"], pk["gn1_b"], pk["eps1"], True)
    h1 = Conv3x3Fn.apply(y, pk["w1"], pb["w1"], pk["b1"], emb_rows, None)
    y2 = _gn(h1, pk["gn2_w"], pk["gn2_b"], pk["eps2"], True)
    if "ws" in pk:
        res = linear(CastBF16.apply(x).reshape(B * H * W, Cin), pk["ws"], pb["ws"], pk["bs"]).reshape(B, H, W, -1)
    else:
        res = x
    return Conv3x3Fn.apply(y2, pk["w2"], pb["w2"], pk["b2"], None, res.contiguous())


def _ln(block: BasicTransformerBlock, name: str, x: torch.Tensor) -> torch.Tensor:
    w, b, eps = block.packed()[name]
    return LayerNormFn.apply(x, w, b, eps, torch.bfloat16)


def transformer_block_train(block: BasicTransformerBlock, t: torch.Tensor, B: int, N: int,
                            ctx_k: Optional[torch.Tensor], ctx_v: Optional[torch.Tensor],
                            key_mask: Optional[torch.Tensor] = None) -> torch.Tensor:
    """BasicTransformerBlock._forward (attention.py:275-285) with grad; t fp32 [B*N, C]; ctx_* fp32 [B, nk, 768];
    key_mask: uint8 [B, N] self-attention key mask (attn1 only, :277) or None."""
    a1, a2, ff = block.attn1, block.attn2, block.ff
    h, d = a1.heads, a1.dim_head
    dp = head_pad(d)
    p1, b1 = a1.packed(), bwd_packs(a1)
    ln1 = _ln(block, "norm1", t)
    qk = linear(ln1, p1["wqk"], b1["wqk"], out_dtype=torch.bfloat16)
    v = linear(ln1, p1["wv"], b1["wv"], out_dtype=torch.bfloat16)
    o = AttentionFn.apply(qk, qk[:, h * dp:], v, B, h, d, N, N, N, key_mask)
    x1 = linear(o, p1["wo"], b1["wo"], p1["bo"], residual=t)
    p2, b2 = a2.packed(), bwd_packs(a2)
    ln2 = _ln(block, "norm2", x1)
    q = linear(ln2, p2["wq"], b2["wq"], out_dtype=torch.bfloat16)
    nk = ctx_k.shape[1]
    nkp = (nk + 7) // 8 * 8
    pad = lambda c: torch.nn.functional.pad(c, (0, 0, 0, nkp - nk)).reshape(B * nkp, c.shape[-1])
    ckb = CastBF16.apply(pad(ctx_k))
    cvb = ckb if ctx_v is ctx_k else CastBF16.apply(pad(ctx_v))
    kc = linear(ckb, p2["wk"], b2["wk"], out_dtype=torch.bfloat16)
    vc = linear(cvb, p2["wv"], b2["wv"], out_dtype=torch.bfloat16)
    o2 = AttentionFn.apply(q, kc, vc, B, h, d, N, nk, nkp)
    x2 = linear(o2, p2["wo"], b2["wo"], p2["bo"], residual=x1)
    pf, bf_ = ff.packed(), bwd_packs(ff)
    ln3 = _ln(block, "norm3", x2)
    proj = linear(ln3, bf_["w1_plain"], bf_["w1"], bf_["b1_plain"], out_dtype=torch.bfloat16)
    hid = GegluFn.apply(proj)
    return linear(hid, pf["w2"], bf_["w2"], pf["b2"], residual=x2)


def spatial_transformer_train(st: SpatialTransformer, x: torch.Tensor, ctx,
                              key_mask: Optional[torch.Tensor] = None) -> torch.Tensor:
    """SpatialTransformer.forward (attention.py:321-341) with grad; x fp32 NHWC; ctx = (v_ctx, k_ctx) fp32 [B,nk,768];
    key_mask: uint8 [B, H*W] (the image mask at this layer's resolution, :332) or None."""
    pk, pb = st.packed(), bwd_packs(st)
    B, H, W, C = x.shape
    T = B * H * W
    xn = _gn(x, pk["gn_w"], pk["gn_b"], pk["gn_eps"], False)
    t = linear(xn.reshape(T, C), pk["w_in"], pb["w_in"], pk["b_in"])
    v_ctx, k_ctx = ctx
    tb = transformer_block_train(st.transformer_blocks[0], t, B, H * W, k_ctx, v_ctx, key_mask)
    out = linear(CastBF16.apply(tb), pk["w_out"], pb["w_out"], pk["b_out"], residual=x.reshape(T, C).contiguous())
    return out.reshape(B, H, W, C)


def unet_forward_train(unet: UNetModel, x: torch.Tensor, timesteps: torch.Tensor, context: torch.Tensor,
                       extra_info: dict) -> torch.Tensor:
    """UNetModel.forward (openaimodel.py:827-1052) with grad w.r.t. `context` [16*B, nk, 768].
    Returns eps fp32 NCHW [B, 4, H, W].  extra_info["img_mask"]: None or float / bool [B, 1, H, W] at the latent's
    resolution; every self-attention layer masks the keys of its nearest-resized copy (attention.py:332 -> :277, as
    the inference path does).  Attention capture and conv attention are not part of the zero-shot distillation branch
    (ddpm.py:3010-3013) and raise."""
    if not extra_info.get("use_layerwise_context", False):
        raise ValueError("extra_info['use_layerwise_context'] must be True")
    if extra_info.get("capture_distill_attn", False):
        raise NotImplementedError("training step: capture_distill_attn")
    if extra_info.get("use_conv_attn_kernel_size", -1) > 0 and extra_info.get("placeholder2indices", None) is not None:
        raise NotImplementedError("training step: the backward of conv attention is not built (zero-shot distillation runs "
                                  "with use_conv_attn_kernel_size = -1)")
    img_mask = extra_info.get("img_mask", None)
    if img_mask is not None:
        check_image_mask(img_mask, x, "extra_info['img_mask']")
    iter_type = extra_info.get("iter_type", "normal_recon")
    pk = unet.packed()
    B = x.shape[0]
    key_masks = {}

    def key_mask(H, W):
        """uint8 [B, H*W] key mask of a self-attention layer at H x W (attention.py:435-437), built once per resolution."""
        if img_mask is None:
            return None
        km = key_masks.get((H, W))
        if km is None:
            m2 = torch.nn.functional.interpolate(img_mask.float(), size=(H, W), mode="nearest")
            km = key_masks[(H, W)] = m2.reshape(B, H * W).bool().to(torch.uint8).contiguous()
        return km
    with torch.no_grad():
        _, rows = unet.time_embedding(timesteps)
    offs = pk["emb_offs"]
    ctx_layers = context.reshape(B, 16, -1, context.shape[-1]).permute(1, 0, 2, 3)          # :866

    def layer_ctx(layer_idx):
        c = ctx_layers[L2CA[layer_idx]]
        if iter_type == "mix_hijk":                                                        # :885-892
            v_c, k_c = c.chunk(2, dim=1)
            return v_c.contiguous(), k_c.contiguous()
        return c, c

    def run(module: TimestepEmbedSequential, h, layer_idx):
        for layer in module:
            if isinstance(layer, ResBlock):
                o, n = offs[id(layer)]
                h = resblock_train(layer, h, rows[:, o:o + n])
            elif isinstance(layer, SpatialTransformer):
                h = spatial_transformer_train(layer, h, layer_ctx(layer_idx), key_mask(h.shape[1], h.shape[2]))
            elif isinstance(layer, Upsample):
                h = UpsampleConvFn.apply(h, layer.packed()["w"], bwd_packs(layer)["w"], layer.packed()["b"])
            elif isinstance(layer, Downsample):
                h = DownsampleConvFn.apply(h, layer.packed()["w"], bwd_packs(layer)["w"], layer.packed()["b"])
            elif isinstance(layer, ConvIn):
                with torch.no_grad():
                    h = layer._run(h)
            else:
                raise NotImplementedError(type(layer))
        return h

    hs = []
    h = x
    layer_idx = 0
    for module in unet.input_blocks:
        h = run(module, h, layer_idx)
        hs.append(h)
        layer_idx += 1
    h = run(unet.middle_block, h, layer_idx)
    layer_idx += 1
    for module in unet.output_blocks:
        h = run(module, torch.cat([h, hs.pop()], dim=-1), layer_idx)
        layer_idx += 1
    y = _gn(h, pk["out_gn_w"], pk["out_gn_b"], pk["out_eps"], True)
    w_f32 = unet.out[2].weight.detach().float().contiguous()
    return ConvOutFn.apply(y, pk["out_w"], pk["out_b"], w_f32, unet.out_channels)


def distill_loss(eps: torch.Tensor, teacher_eps: torch.Tensor, num_denoising_steps: int = 1) -> torch.Tensor:
    """Whole-image MSE against the teacher's noise (calc_recon_loss ddpm.py:3571-3595 with no masks, :3010-3013),
    scaled by 1/sqrt(steps) (:3037)."""
    return torch.nn.functional.mse_loss(eps, teacher_eps) / math.sqrt(num_denoising_steps)


def check_image_mask(mask, x: torch.Tensor, name: str) -> None:
    """An image / face mask of the latent batch x [B, C, H, W]: a float or bool tensor [B, 1, H, W] on x's device."""
    if not isinstance(mask, torch.Tensor):
        raise ValueError(f"{name}: expected a tensor, got {type(mask).__name__}")
    if not (mask.dtype == torch.bool or mask.dtype.is_floating_point):
        raise ValueError(f"{name}: expected a float or bool tensor, got {mask.dtype}")
    want = (x.shape[0], 1, x.shape[2], x.shape[3])
    if tuple(mask.shape) != want:
        raise ValueError(f"{name}: expected shape {want} (the latent's batch and resolution), got {tuple(mask.shape)}")
    if mask.device != x.device:
        raise ValueError(f"{name}: on {mask.device}, the latents are on {x.device}")


def calc_recon_loss(eps: torch.Tensor, target: torch.Tensor, img_mask: Optional[torch.Tensor] = None,
                    fg_mask: Optional[torch.Tensor] = None, fg_pixel_weight: float = 1.,
                    bg_pixel_weight: float = 1.) -> torch.Tensor:
    """Masked, foreground / background weighted MSE of calc_recon_loss (ddpm.py:3571-3595), restated:
        pix = (eps*img - target*img)^2,  wf = fg*img*fg_pixel_weight,  wb = (1 - fg)*img*bg_pixel_weight,
        loss = (sum pix*wf + sum pix*wb) / (sum wf + sum wb)
    with the [B, 1, H, W] masks broadcast over the channels of eps / target [B, C, H, W]; a missing mask is all ones, so
    with neither mask this is F.mse_loss.  Parity unpinned: no reference outputs exist to pin this restatement to (as
    for tests/vae_encoder_oracle.py).  The reference's call-site weights are not restated; callers pass their own
    (DistillStep: fg_pixel_weight / bg_pixel_weight, default 1).  Plain tensor arithmetic, no host read-back."""
    ones = torch.ones_like(eps[:, :1])
    img = ones if img_mask is None else img_mask.to(eps.dtype)
    fg = ones if fg_mask is None else fg_mask.to(eps.dtype)
    pix = (eps * img - target * img) ** 2
    wf = (fg * img * fg_pixel_weight).expand_as(eps)
    wb = ((1 - fg) * img * bg_pixel_weight).expand_as(eps)
    return ((pix * wf).sum() + (pix * wb).sum()) / (wf.sum() + wb.sum())


class GraphedUNetLoss:
    """loss = distill_loss(UNet(x_noisy, t, c), teacher_eps) and dloss/dc replayed from ONE CUDA graph.

    The UNet is frozen (ddpm.py:783-786), so the ~3500 kernel launches of its forward and backward-to-context depend
    only on the shapes: they are captured once per geometry (static input / output buffers, torch.autograd.grad inside
    the capture) and replayed per micro-batch - the host-side launch gaps of the eager tape (a fifth of the step)
    disappear.  Weights are read through the version-keyed packs, so a repack invalidates the capture.
    With an image and / or face mask the loss is calc_recon_loss with the given pixel weights and the image mask also
    masks the UNet's self-attention keys; the masks are static buffers of the capture, and the geometry key records
    which of them are present, so masked and unmasked micro-batches never share a graph."""

    def __init__(self, unet: UNetModel, extra_info: dict, fg_pixel_weight: float = 1., bg_pixel_weight: float = 1.):
        self.unet, self.extra_info = unet, dict(extra_info)
        self.fg_pixel_weight, self.bg_pixel_weight = fg_pixel_weight, bg_pixel_weight
        self._g = {}

    def _build(self, x, t, c, teacher, img_mask, fg_mask):
        from .attention import PackedModule
        st = {"x": x.clone(), "t": t.clone(), "c": c.clone().requires_grad_(True), "teacher": teacher.clone(),
              "img_mask": None if img_mask is None else img_mask.clone(),
              "fg_mask": None if fg_mask is None else fg_mask.clone()}

        def run():
            extra = dict(self.extra_info)
            if st["img_mask"] is not None:
                extra["img_mask"] = st["img_mask"]
            eps = unet_forward_train(self.unet, st["x"], st["t"], st["c"], extra)
            if st["img_mask"] is None and st["fg_mask"] is None:
                loss = distill_loss(eps, st["teacher"])
            else:
                loss = calc_recon_loss(eps, st["teacher"], st["img_mask"], st["fg_mask"], self.fg_pixel_weight,
                                       self.bg_pixel_weight)
            (gc,) = torch.autograd.grad(loss, st["c"])
            return loss.detach(), gc

        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                run()
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            st["loss"], st["grad_c"] = run()
        st["graph"], st["epoch"] = graph, PackedModule.PACK_EPOCH
        return st

    def __call__(self, x_noisy, t, c, teacher_eps, img_mask=None, fg_mask=None):
        from .attention import PackedModule
        for name, m in (("img_mask", img_mask), ("fg_mask", fg_mask)):
            if m is not None:
                check_image_mask(m, x_noisy, name)
        key = (tuple(x_noisy.shape), tuple(c.shape), t.dtype,
               None if img_mask is None else img_mask.dtype, None if fg_mask is None else fg_mask.dtype)
        st = self._g.get(key)
        if st is None or st["epoch"] != PackedModule.PACK_EPOCH:
            st = self._g[key] = self._build(x_noisy, t, c, teacher_eps, img_mask, fg_mask)
        st["x"].copy_(x_noisy)
        st["t"].copy_(t)
        st["teacher"].copy_(teacher_eps)
        for name, m in (("img_mask", img_mask), ("fg_mask", fg_mask)):
            if m is not None:
                st[name].copy_(m)
        with torch.no_grad():
            st["c"].copy_(c)
        st["graph"].replay()
        return st["loss"].clone(), st["grad_c"].clone()
