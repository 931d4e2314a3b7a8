"""Host mirror of the first stage: latents -> RGB (decoder) and, with `with_encoder=True`, RGB -> posterior over latents
(encoder, for img2img) - SURVEY.md section 8(f) row N1.

Reference: ldm/modules/diffusionmodules/model.py (ResnetBlock :83-142, AttnBlock :151-242, Upsample :43-58,
Downsample :61-79, Encoder :408-500, Decoder :502-609), ldm/modules/distributions/distributions.py
(DiagonalGaussianDistribution :24-44), ldm/models/autoencoder.py (AutoencoderKL :285-333) and
LatentDiffusion.decode_first_stage / encode_first_stage / get_first_stage_encoding (ldm/models/diffusion/ddpm.py,
the `1/scale_factor` scaling :1267), configured by configs/stable-diffusion/v1-inference-ada.yaml:53-73 (ch 128,
ch_mult [1,2,4,4], 2 res blocks, z_channels 4, double_z, no attention except the single-head 512-channel AttnBlock in
the middle).

Same constructor arguments, forward signatures and state_dict key names as the reference (`encoder.*`, `decoder.*`,
`quant_conv.*`, `post_quant_conv.*`), so an SD-1.5 VAE checkpoint loads unchanged.  By default only the decode side is
built (the sampling path): the encoder / quant_conv keys of a full checkpoint are then ignored, and the loss keys always
are.  The torch.nn layers only hold parameters; all arithmetic runs in
libadaface_b200.so with the same kernels as the UNet: NHWC fp32 residual stream, bf16 tensor-core operands, GroupNorm
statistics produced by the conv epilogues.  The middle AttnBlock has ONE head of 512 channels over h*w tokens - too wide
for the flash kernels' TMEM accumulators - so, like the reference, it materialises the scores: two tcgen05 GEMMs and a
row-softmax kernel per image (34 GFLOP per image, 3 % of the decoder).
"""
from __future__ import annotations

from typing import Optional

import torch
from torch import nn

from . import ops
from .attention import PackedModule
from .packing import pack_conv1x1, pack_conv3x3
from .unet import Act, _conv_out_act, _nchw


def Normalize(in_channels, num_groups=32):
    """model.py:39-40."""
    return nn.GroupNorm(num_groups=num_groups, num_channels=in_channels, eps=1e-6, affine=True)


def _f(t: torch.Tensor) -> torch.Tensor:
    return t.detach().float().contiguous()


class Upsample(PackedModule):
    """model.py:43-58: nearest x2 then conv3x3."""

    def __init__(self, in_channels, with_conv):
        super().__init__()
        if not with_conv:
            raise NotImplementedError("Upsample: resamp_with_conv=False is not used by the SD-1.5 VAE")
        self.with_conv = with_conv
        self.conv = nn.Conv2d(in_channels, in_channels, kernel_size=3, stride=1, padding=1)

    def _pack(self):
        return {"w": pack_conv3x3(self.conv.weight.detach()), "b": _f(self.conv.bias)}

    def _run(self, a: Act) -> Act:
        pk = self.packed()
        x = a.t
        B, H, W, C = x.shape
        up = torch.empty(B, 2 * H, 2 * W, C, dtype=torch.bfloat16, device=x.device)
        ops.upsample2x_cast(x, up)
        out, st = _conv_out_act(B, 2 * H, 2 * W, C, x.device)
        ops.conv3x3(up, pk["w"], out, bias=pk["b"], gn_stats=st.buf if st else None)
        return Act(out, st)

    def forward(self, x):
        return _nchw(self._run(Act(x.float().permute(0, 2, 3, 1).contiguous())).t)


class Downsample(PackedModule):
    """model.py:61-79: F.pad(x, (0, 1, 0, 1)) then conv3x3 stride 2 pad 0 - one kernel, the pad is TMA zero fill."""

    def __init__(self, in_channels, with_conv):
        super().__init__()
        if not with_conv:
            raise NotImplementedError("Downsample: resamp_with_conv=False (avg_pool2d) is not used by the SD-1.5 VAE")
        self.with_conv = with_conv
        self.conv = nn.Conv2d(in_channels, in_channels, kernel_size=3, stride=2, padding=0)

    def _pack(self):
        return {"w": pack_conv3x3(self.conv.weight.detach()), "b": _f(self.conv.bias)}

    def _run(self, a: Act) -> Act:
        pk = self.packed()
        x = a.t
        B, H, W, C = x.shape
        xb = ops.cast_bf16(x)
        out, st = _conv_out_act(B, H // 2, W // 2, C, x.device)
        ops.conv3x3_down01(xb, pk["w"], out, bias=pk["b"], gn_stats=st.buf if st else None)
        return Act(out, st)

    def forward(self, x):
        return _nchw(self._run(Act(x.float().permute(0, 2, 3, 1).contiguous())).t)


class ResnetBlock(PackedModule):
    """model.py:83-142 without a timestep embedding (Decoder.temb_ch = 0, :511)."""

    def __init__(self, *, in_channels, out_channels=None, conv_shortcut=False, dropout, temb_channels=512):
        super().__init__()
        if conv_shortcut:
            raise NotImplementedError("ResnetBlock: conv_shortcut=True is not used by the SD-1.5 VAE")
        self.in_channels = in_channels
        out_channels = in_channels if out_channels is None else out_channels
        self.out_channels = out_channels
        self.use_conv_shortcut = conv_shortcut
        self.norm1 = Normalize(in_channels)
        self.conv1 = nn.Conv2d(in_channels, out_channels, kernel_size=3, stride=1, padding=1)
        if temb_channels > 0:
            self.temb_proj = nn.Linear(temb_channels, out_channels)
        self.norm2 = Normalize(out_channels)
        self.dropout = nn.Dropout(dropout)
        self.conv2 = nn.Conv2d(out_channels, out_channels, kernel_size=3, stride=1, padding=1)
        if self.in_channels != self.out_channels:
            self.nin_shortcut = nn.Conv2d(in_channels, out_channels, kernel_size=1, stride=1, padding=0)

    def _pack(self):
        pk = {"n1w": _f(self.norm1.weight), "n1b": _f(self.norm1.bias), "eps1": float(self.norm1.eps),
              "w1": pack_conv3x3(self.conv1.weight.detach()), "b1": _f(self.conv1.bias),
              "n2w": _f(self.norm2.weight), "n2b": _f(self.norm2.bias), "eps2": float(self.norm2.eps),
              "w2": pack_conv3x3(self.conv2.weight.detach()), "b2": _f(self.conv2.bias)}
        if self.in_channels != self.out_channels:
            pk["ws"] = pack_conv1x1(self.nin_shortcut.weight.detach())
            pk["bs"] = _f(self.nin_shortcut.bias)
        return pk

    def _run(self, a: Act) -> Act:
        pk = self.packed()
        x = a.t
        B, H, W, Cin = x.shape
        assert Cin == self.in_channels, (Cin, self.in_channels)
        Cout, dev = self.out_channels, x.device
        has_nin = "ws" in pk
        y = torch.empty(B, H, W, Cin, dtype=torch.bfloat16, device=dev)
        raw = torch.empty(B, H, W, Cin, dtype=torch.bfloat16, device=dev) if has_nin else None
        ops.groupnorm_apply(x, a.stats(), pk["n1w"], pk["n1b"], pk["eps1"], True, y, raw=raw)        # :124-126
        h1, st1 = _conv_out_act(B, H, W, Cout, dev)
        ops.conv3x3(y, pk["w1"], h1, bias=pk["b1"], gn_stats=st1.buf if st1 else None)               # :127
        del y
        y2 = torch.empty(B, H, W, Cout, dtype=torch.bfloat16, device=dev)
        ops.groupnorm_apply(h1, st1 if st1 else ops.groupnorm_stats(h1), pk["n2w"], pk["n2b"], pk["eps2"], True,
                            y2)                                                                      # :132-133
        del h1
        if has_nin:
            res = torch.empty(B, H, W, Cout, dtype=torch.float32, device=dev)
            ops.gemm(raw.reshape(B * H * W, Cin), pk["ws"], res, bias=pk["bs"])                      # :140
        else:
            res = x
        out, sto = _conv_out_act(B, H, W, Cout, dev)
        ops.conv3x3(y2, pk["w2"], out, bias=pk["b2"], residual=res, gn_stats=sto.buf if sto else None)  # :135,:142
        return Act(out, sto)

    def forward(self, x, temb):
        if temb is not None:
            raise NotImplementedError("ResnetBlock: timestep embeddings are not used by the VAE decoder (temb_ch = 0)")
        return _nchw(self._run(Act(x.float().permute(0, 2, 3, 1).contiguous())).t)


class AttnBlock(PackedModule):
    """model.py:151-242: single-head self-attention over h*w tokens with c channels, scores materialised."""

    def __init__(self, in_channels):
        super().__init__()
        self.in_channels = in_channels
        self.norm = Normalize(in_channels)
        self.q = nn.Conv2d(in_channels, in_channels, kernel_size=1, stride=1, padding=0)
        self.k = nn.Conv2d(in_channels, in_channels, kernel_size=1, stride=1, padding=0)
        self.v = nn.Conv2d(in_channels, in_channels, kernel_size=1, stride=1, padding=0)
        self.proj_out = nn.Conv2d(in_channels, in_channels, kernel_size=1, stride=1, padding=0)

    def _pack(self):
        C = self.in_channels
        wp = self.proj_out.weight.detach().float().reshape(C, C)
        # softmax rows sum to one, so attn @ (V + 1 b_v^T) = attn @ V + b_v: the value bias moves behind proj_out
        bp = self.proj_out.bias.detach().float() + wp @ self.v.bias.detach().float()
        return {"nw": _f(self.norm.weight), "nb": _f(self.norm.bias), "eps": float(self.norm.eps),
                "wq": pack_conv1x1(self.q.weight.detach()), "bq": _f(self.q.bias),
                "wk": pack_conv1x1(self.k.weight.detach()), "bk": _f(self.k.bias),
                "wv": pack_conv1x1(self.v.weight.detach()),
                "wp": pack_conv1x1(self.proj_out.weight.detach()), "bp": bp.contiguous()}

    def _run(self, a: Act) -> Act:
        pk = self.packed()
        x = a.t
        B, H, W, C = x.shape
        N, dev = H * W, x.device
        if N % 8 != 0:
            raise ValueError(f"AttnBlock: h*w = {N} must be a multiple of 8")
        y = torch.empty(B * N, C, dtype=torch.bfloat16, device=dev)
        ops.groupnorm_apply(x, a.stats(), pk["nw"], pk["nb"], pk["eps"], False, y.view(B, H, W, C))    # :181
        q = torch.empty(B * N, C, dtype=torch.bfloat16, device=dev)
        k = torch.empty(B * N, C, dtype=torch.bfloat16, device=dev)
        ops.gemm(y, pk["wq"], q, bias=pk["bq"])                                                        # :182
        ops.gemm(y, pk["wk"], k, bias=pk["bk"])                                                        # :183
        o = torch.empty(B * N, C, dtype=torch.bfloat16, device=dev)
        s = torch.empty(N, N, dtype=torch.float32, device=dev)
        p = torch.empty(N, N, dtype=torch.bfloat16, device=dev)
        vt = torch.empty(C, N, dtype=torch.bfloat16, device=dev)
        scale = float(int(C) ** (-0.5))
        for b in range(B):
            rows = slice(b * N, (b + 1) * N)
            ops.gemm(pk["wv"], y[rows], vt)                    # V^T [c, hw] = W_v . Y_b^T (bias folded into bp)     :184
            ops.gemm(q[rows], k[rows], s)                      # w_[i, j] = sum_c q[i, c] k[j, c]                    :190
            ops.softmax_rows(s, scale, p)                      # * c^-1/2, softmax over j                            :192-193
            ops.gemm(p, vt, o[rows])                           # h_[i, c] = sum_j w_[i, j] v[j, c]                   :236-238
        out = torch.empty(B, H, W, C, dtype=torch.float32, device=dev)
        st = ops.gn_stats_for_gemm(B, N, C, dev)
        ops.gemm(o, pk["wp"], out.view(B * N, C), bias=pk["bp"], residual=x.view(B * N, C),
                 gn_stats=st.buf if st else None)                                                      # :240-242
        return Act(out, st)

    def forward(self, x, mask=None):
        if mask is not None:
            raise NotImplementedError("AttnBlock: fg/bg pair masks belong to the training encoder path")
        return _nchw(self._run(Act(x.float().permute(0, 2, 3, 1).contiguous())).t)


def make_attn(in_channels, attn_type="vanilla"):
    """model.py:245-253."""
    assert attn_type in ["vanilla", "linear", "none"], f"attn_type {attn_type} unknown"
    if attn_type == "vanilla":
        return AttnBlock(in_channels)
    if attn_type == "none":
        return nn.Identity(in_channels)
    raise NotImplementedError("LinAttnBlock is not used by the SD-1.5 VAE")


class _ConvIn(nn.Conv2d):
    """Decoder.conv_in (4 -> 512) / Encoder.conv_in (3 -> 128): reads the public NCHW input, writes the NHWC fp32
    stream."""

    def _run(self, z_nchw: torch.Tensor) -> torch.Tensor:
        B, C, H, W = z_nchw.shape
        out = torch.empty(B, H, W, self.out_channels, dtype=torch.float32, device=z_nchw.device)
        return ops.conv_in(z_nchw.float().contiguous(), _f(self.weight), _f(self.bias), out)


class Decoder(PackedModule):
    """model.py:502-609."""

    def __init__(self, *, ch, out_ch, ch_mult=(1, 2, 4, 8), num_res_blocks, attn_resolutions, dropout=0.0,
                 resamp_with_conv=True, in_channels, resolution, z_channels, give_pre_end=False, tanh_out=False,
                 use_linear_attn=False, attn_type="vanilla", **ignorekwargs):
        super().__init__()
        if use_linear_attn:
            attn_type = "linear"
        if z_channels != 4 or out_ch > 4:
            raise NotImplementedError("Decoder: z_channels must be 4 and out_ch <= 4 (SD-1.5 VAE)")
        self.ch = ch
        self.temb_ch = 0
        self.num_resolutions = len(ch_mult)
        self.num_res_blocks = num_res_blocks
        self.resolution = resolution
        self.in_channels = in_channels
        self.out_ch = out_ch
        self.give_pre_end = give_pre_end
        self.tanh_out = tanh_out
        block_in = ch * ch_mult[self.num_resolutions - 1]
        curr_res = resolution // 2 ** (self.num_resolutions - 1)
        self.z_shape = (1, z_channels, curr_res, curr_res)
        self.conv_in = _ConvIn(z_channels, block_in, kernel_size=3, stride=1, padding=1)
        self.mid = nn.Module()
        self.mid.block_1 = ResnetBlock(in_channels=block_in, out_channels=block_in, temb_channels=self.temb_ch,
                                       dropout=dropout)
        self.mid.attn_1 = make_attn(block_in, attn_type=attn_type)
        self.mid.block_2 = ResnetBlock(in_channels=block_in, out_channels=block_in, temb_channels=self.temb_ch,
                                       dropout=dropout)
        self.up = nn.ModuleList()
        for i_level in reversed(range(self.num_resolutions)):
            block = nn.ModuleList()
            attn = nn.ModuleList()
            block_out = ch * ch_mult[i_level]
            for _ in range(self.num_res_blocks + 1):
                block.append(ResnetBlock(in_channels=block_in, out_channels=block_out, temb_channels=self.temb_ch,
                                         dropout=dropout))
                block_in = block_out
                if curr_res in attn_resolutions:
                    attn.append(make_attn(block_in, attn_type=attn_type))
            up = nn.Module()
            up.block = block
            up.attn = attn
            if i_level != 0:
                up.upsample = Upsample(block_in, resamp_with_conv)
                curr_res = curr_res * 2
            self.up.insert(0, up)  # prepend to get consistent order
        self.norm_out = Normalize(block_in)
        self.conv_out = nn.Conv2d(block_in, out_ch, kernel_size=3, stride=1, padding=1)

    def _pack(self):
        # conv_out: Cout 3 padded to 8 zero rows for the tensor-core conv (like the UNet's 320 -> 4 out conv)
        w = self.conv_out.weight.detach()
        wp = torch.zeros(8, *w.shape[1:], dtype=w.dtype, device=w.device)
        wp[:w.shape[0]] = w
        bp = torch.zeros(8, dtype=torch.float32, device=w.device)
        bp[:w.shape[0]] = self.conv_out.bias.detach().float()
        return {"nw": _f(self.norm_out.weight), "nb": _f(self.norm_out.bias), "eps": float(self.norm_out.eps),
                "w": pack_conv3x3(wp), "b": bp}

    def forward(self, z):
        """z: [B, z_channels, h, w] (any float dtype) -> [B, out_ch, 8h, 8w] fp32 NCHW."""
        if not z.is_cuda:
            raise RuntimeError("Decoder: the B200 path has no CPU fallback - move the latents to a CUDA device")
        self.last_z_shape = z.shape
        pk = self.packed()
        h = Act(self.conv_in._run(z))                                        # :583
        h = self.mid.block_1._run(h)                                         # :586
        if isinstance(self.mid.attn_1, AttnBlock):
            h = self.mid.attn_1._run(h)                                      # :587
        h = self.mid.block_2._run(h)                                         # :588
        for i_level in reversed(range(self.num_resolutions)):                # :591-597
            for i_block in range(self.num_res_blocks + 1):
                h = self.up[i_level].block[i_block]._run(h)
                if len(self.up[i_level].attn) > 0:
                    h = self.up[i_level].attn[i_block]._run(h)
            if i_level != 0:
                h = self.up[i_level].upsample._run(h)
        if self.give_pre_end:
            return _nchw(h.t)
        B, H, W, C = h.t.shape
        dev = h.t.device
        y = torch.empty(B, H, W, C, dtype=torch.bfloat16, device=dev)
        ops.groupnorm_apply(h.t, h.stats(), pk["nw"], pk["nb"], pk["eps"], True, y)    # :603-604
        del h
        o8 = torch.empty(B, H, W, 8, dtype=torch.float32, device=dev)
        ops.conv3x3(y, pk["w"], o8, bias=pk["b"], bn=64)                                # :605
        out = torch.empty(B, self.out_ch, H, W, dtype=torch.float32, device=dev)
        ops.nhwc_to_nchw(o8, out)
        if self.tanh_out:
            out = torch.tanh(out)
        return out


class Encoder(PackedModule):
    """model.py:408-500."""

    def __init__(self, *, ch, out_ch, ch_mult=(1, 2, 4, 8), num_res_blocks, attn_resolutions, dropout=0.0,
                 resamp_with_conv=True, in_channels, resolution, z_channels, double_z=True, use_linear_attn=False,
                 attn_type="vanilla", **ignore_kwargs):
        super().__init__()
        if use_linear_attn:
            attn_type = "linear"
        self.ch = ch
        self.temb_ch = 0
        self.num_resolutions = len(ch_mult)
        self.num_res_blocks = num_res_blocks
        self.resolution = resolution
        self.in_channels = in_channels
        self.conv_in = _ConvIn(in_channels, self.ch, kernel_size=3, stride=1, padding=1)
        curr_res = resolution
        in_ch_mult = (1,) + tuple(ch_mult)
        self.in_ch_mult = in_ch_mult
        self.down = nn.ModuleList()
        for i_level in range(self.num_resolutions):
            block = nn.ModuleList()
            attn = nn.ModuleList()
            block_in = ch * in_ch_mult[i_level]
            block_out = ch * ch_mult[i_level]
            for _ in range(self.num_res_blocks):
                block.append(ResnetBlock(in_channels=block_in, out_channels=block_out, temb_channels=self.temb_ch,
                                         dropout=dropout))
                block_in = block_out
                if curr_res in attn_resolutions:
                    attn.append(make_attn(block_in, attn_type=attn_type))
            down = nn.Module()
            down.block = block
            down.attn = attn
            if i_level != self.num_resolutions - 1:
                down.downsample = Downsample(block_in, resamp_with_conv)
                curr_res = curr_res // 2
            self.down.append(down)
        self.mid = nn.Module()
        self.mid.block_1 = ResnetBlock(in_channels=block_in, out_channels=block_in, temb_channels=self.temb_ch,
                                       dropout=dropout)
        self.mid.attn_1 = make_attn(block_in, attn_type=attn_type)
        self.mid.block_2 = ResnetBlock(in_channels=block_in, out_channels=block_in, temb_channels=self.temb_ch,
                                       dropout=dropout)
        self.norm_out = Normalize(block_in)
        self.conv_out = nn.Conv2d(block_in, 2 * z_channels if double_z else z_channels, kernel_size=3, stride=1,
                                  padding=1)
        if self.conv_out.out_channels % 8:
            raise NotImplementedError("Encoder: conv_out needs a multiple of 8 output channels (double_z, z_channels 4)")

    def _pack(self):
        return {"nw": _f(self.norm_out.weight), "nb": _f(self.norm_out.bias), "eps": float(self.norm_out.eps),
                "w": pack_conv3x3(self.conv_out.weight.detach()), "b": _f(self.conv_out.bias)}

    def _run(self, x: torch.Tensor, head=None) -> torch.Tensor:
        """x NCHW [B, in_channels, H, W] -> conv_out output NHWC fp32 [B, H/8, W/8, Cout].  head = (packed weight, bias)
        replaces conv_out's own (AutoencoderKL folds quant_conv into it)."""
        if not x.is_cuda:
            raise RuntimeError("Encoder: the B200 path has no CPU fallback - move the images to a CUDA device")
        pk = self.packed()
        h = Act(self.conv_in._run(x))                                        # :470
        for i_level in range(self.num_resolutions):                          # :471-478
            for i_block in range(self.num_res_blocks):
                h = self.down[i_level].block[i_block]._run(h)
                if len(self.down[i_level].attn) > 0:
                    h = self.down[i_level].attn[i_block]._run(h)
            if i_level != self.num_resolutions - 1:
                h = self.down[i_level].downsample._run(h)
        h = self.mid.block_1._run(h)                                         # :482
        if isinstance(self.mid.attn_1, AttnBlock):
            h = self.mid.attn_1._run(h)                                      # :483
        h = self.mid.block_2._run(h)                                         # :484
        B, H, W, C = h.t.shape
        dev = h.t.device
        y = torch.empty(B, H, W, C, dtype=torch.bfloat16, device=dev)
        ops.groupnorm_apply(h.t, h.stats(), pk["nw"], pk["nb"], pk["eps"], True, y)    # :487-488
        del h
        w, b = head if head is not None else (pk["w"], pk["b"])
        out = torch.empty(B, H, W, int(w.shape[0]), dtype=torch.float32, device=dev)
        ops.conv3x3(y, w, out, bias=b, bn=64)                                            # :489
        return out

    def forward(self, x, mask=None):
        """x: [B, in_channels, H, W] -> [B, Cout, H/8, W/8] fp32 NCHW."""
        if mask is not None:
            raise NotImplementedError("Encoder: the fg/bg mask input belongs to the fork's training path")
        return _nchw(self._run(x.float().contiguous()))


class DiagonalGaussianDistribution(object):
    """distributions.py:24-44 over the encoder's moments.  mean and the clamped logvar come out of one kernel
    (af_vae_posterior), which also draws sample() = mean + std * noise - with the noise taken from the host generator
    like the reference (`torch.randn(self.mean.shape)`), so the global CPU RNG stream advances as there.  std, var and
    the NCHW `parameters` are formed on first use.  kl() / nll() are training losses and not mirrored."""

    def __init__(self, parameters=None, deterministic=False, *, moments_nhwc=None):
        if moments_nhwc is None:
            moments_nhwc = parameters.float().permute(0, 2, 3, 1).contiguous()
        self._moments = moments_nhwc
        self._parameters = parameters
        self.deterministic = deterministic
        B, H, W, C2 = moments_nhwc.shape
        zc = C2 // 2
        dev = moments_nhwc.device
        self.mean = torch.empty(B, zc, H, W, dtype=torch.float32, device=dev)
        self.logvar = torch.empty_like(self.mean)
        ops.vae_posterior(moments_nhwc, None, 1.0, self.mean, logvar=self.logvar)
        self._std = self._var = None

    @property
    def parameters(self):
        if self._parameters is None:
            self._parameters = self._moments.permute(0, 3, 1, 2).contiguous()
        return self._parameters

    @property
    def std(self):
        if self._std is None:
            self._std = torch.zeros_like(self.mean) if self.deterministic else torch.exp(0.5 * self.logvar)
        return self._std

    @property
    def var(self):
        if self._var is None:
            self._var = torch.zeros_like(self.mean) if self.deterministic else torch.exp(self.logvar)
        return self._var

    def scaled_sample(self, scale: float = 1.0, noise: Optional[torch.Tensor] = None) -> torch.Tensor:
        """scale * sample() in one kernel: get_first_stage_encoding's scale_factor * z.  noise (NCHW like mean) replaces
        the draw from the host generator."""
        if noise is None:
            noise = torch.randn(self.mean.shape)
        noise = noise.to(device=self.mean.device, dtype=torch.float32).contiguous()
        z = torch.empty_like(self.mean)
        # deterministic: std is 0, so mean + 0 * noise == mean (the reference still draws the noise)
        ops.vae_posterior(self._moments, None if self.deterministic else noise, float(scale), z)
        return z

    def sample(self):
        return self.scaled_sample(1.0)

    def mode(self):
        return self.mean


SD15_VAE_DDCONFIG = dict(  # configs/stable-diffusion/v1-inference-ada.yaml:58-72
    double_z=True, z_channels=4, resolution=256, in_channels=3, out_ch=3, ch=128, ch_mult=[1, 2, 4, 4],
    num_res_blocks=2, attn_resolutions=[], dropout=0.0)


class AutoencoderKL(nn.Module):
    """ldm/models/autoencoder.py:285-333.  Decode side: `post_quant_conv` (1x1, embed_dim -> z_channels) is a tiny fp32
    channel-mix kernel on the NCHW latent (16 MACs per pixel) in front of the decoder's conv_in kernel; the
    `1 / scale_factor` of decode_first_stage rides along as its input scale.  with_encoder=True also builds the encoder
    side: `quant_conv` (1x1, 2*z_channels -> 2*embed_dim) is linear and directly follows the encoder's 3x3 conv_out, so
    it is folded into that convolution's weights (fp32 product, one bf16 rounding) and the moments leave one
    tensor-core conv."""

    def __init__(self, ddconfig=None, lossconfig=None, embed_dim=4, ckpt_path=None, ignore_keys=(), image_key="image",
                 colorize_nlabels=None, monitor=None, with_encoder=False):
        super().__init__()
        ddconfig = dict(SD15_VAE_DDCONFIG if ddconfig is None else ddconfig)
        self.image_key = image_key
        self.embed_dim = embed_dim
        self.with_encoder = with_encoder
        if with_encoder:
            if not ddconfig.get("double_z", True):
                raise NotImplementedError("AutoencoderKL: the encoder needs double_z (autoencoder.py:299)")
            self.encoder = Encoder(**ddconfig)
        self.decoder = Decoder(**ddconfig)
        if with_encoder:
            self.quant_conv = nn.Conv2d(2 * ddconfig["z_channels"], 2 * embed_dim, 1)
        self.post_quant_conv = nn.Conv2d(embed_dim, ddconfig["z_channels"], 1)
        if ckpt_path is not None:
            sd = torch.load(ckpt_path, map_location="cpu")
            self.load_state_dict(sd.get("state_dict", sd))

    def load_state_dict(self, state_dict, strict: bool = True, **kw):
        """Full AutoencoderKL checkpoints also carry loss.* tensors (and encoder.* / quant_conv.*, which only a module
        built with_encoder uses): what this module has no parameter for is dropped instead of failing a strict load."""
        prefixes = ("decoder.", "post_quant_conv.") + (("encoder.", "quant_conv.") if self.with_encoder else ())
        keep = {k: v for k, v in state_dict.items() if k.startswith(prefixes)}
        return super().load_state_dict(keep, strict=strict, **kw)

    def _moments_head(self):
        """conv_out with quant_conv folded in: W' = Wq . Wc, b' = Wq . bc + bq in fp32, then the bf16 pack."""
        co, qc = self.encoder.conv_out, self.quant_conv
        params = (co.weight, co.bias, qc.weight, qc.bias)
        key = tuple((p.data_ptr(), p._version) for p in params)
        ent = self.__dict__.get("_head")
        if ent is None or ent[0] != key:
            with torch.no_grad():
                wq = qc.weight.detach().float().reshape(qc.out_channels, qc.in_channels)
                wc = co.weight.detach().float()
                w = (wq @ wc.reshape(wc.shape[0], -1)).reshape(qc.out_channels, *wc.shape[1:])
                b = wq @ co.bias.detach().float() + qc.bias.detach().float()
            ent = (key, (pack_conv3x3(w), b.contiguous()))
            self.__dict__["_head"] = ent
        return ent[1]

    @torch.no_grad()
    def _moments(self, x) -> torch.Tensor:
        """x NCHW images -> quant_conv(encoder(x)) as NHWC fp32 [B, H/8, W/8, 2*embed_dim]."""
        if not self.with_encoder:
            raise NotImplementedError("AutoencoderKL.encode: build the module with with_encoder=True (the default is the "
                                      "decode side only)")
        if not x.is_cuda:
            raise RuntimeError("AutoencoderKL.encode: the B200 path has no CPU fallback - move the images to a CUDA device")
        return self.encoder._run(x.float().contiguous(), head=self._moments_head())

    def encode(self, x, mask=None):
        """autoencoder.py:316-320: NCHW images in [-1, 1] -> DiagonalGaussianDistribution over the latents."""
        if mask is not None:
            raise NotImplementedError("AutoencoderKL.encode: the fg/bg mask input belongs to the fork's training path")
        return DiagonalGaussianDistribution(moments_nhwc=self._moments(x))

    @torch.no_grad()
    def decode(self, z, in_scale: float = 1.0):
        if not z.is_cuda:
            raise RuntimeError("AutoencoderKL.decode: the B200 path has no CPU fallback - move the latents to a CUDA device")
        pq = self.post_quant_conv
        w = pq.weight.detach().float().reshape(pq.out_channels, -1).contiguous()
        z = ops.channel_mix4(z.float().contiguous(), w, pq.bias.detach().float().contiguous(), in_scale)   # :331
        return self.decoder(z)                                                                              # :332

    def forward(self, z):
        return self.decode(z)


def encode_first_stage(first_stage_model: AutoencoderKL, x: torch.Tensor, max_batch: Optional[int] = None
                       ) -> DiagonalGaussianDistribution:
    """LatentDiffusion.encode_first_stage (ddpm.py, the non-split branch): first_stage_model.encode(x).  max_batch bounds
    the images encoded per pass (a 512^2 activation with 128 channels is 134 MB per image and tensor)."""
    if max_batch is None or x.shape[0] <= max_batch:
        return first_stage_model.encode(x)
    return DiagonalGaussianDistribution(moments_nhwc=torch.cat(
        [first_stage_model._moments(x[i:i + max_batch]) for i in range(0, x.shape[0], max_batch)], 0))


def decode_first_stage(first_stage_model: AutoencoderKL, z: torch.Tensor, scale_factor: float = 0.18215,
                       max_batch: Optional[int] = None) -> torch.Tensor:
    """LatentDiffusion.decode_first_stage (ddpm.py:1260-1318, the non-split branch): z / scale_factor -> decode.
    max_batch bounds the images decoded per pass (activations at 512^2 are 1 GB per 8 images and tensor)."""
    s = 1. / scale_factor                                                     # :1267 (applied inside the first kernel)
    if max_batch is None or z.shape[0] <= max_batch:
        return first_stage_model.decode(z, in_scale=s)
    return torch.cat([first_stage_model.decode(z[i:i + max_batch], in_scale=s) for i in range(0, z.shape[0], max_batch)], 0)
