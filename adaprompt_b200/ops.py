"""Thin tensor-level wrappers over the C ABI (one function per af_* entry point).

PyTorch is plumbing here: it owns device memory and streams; all arithmetic happens in
libadaface_b200.so.  Every wrapper validates dtype/device/contiguity, passes raw pointers and
raises on a non-zero return code.  No op has a CPU or eager fallback.
"""
from __future__ import annotations

from ctypes import byref
from typing import Optional

import torch

from . import _lib
from ._lib import AF_DTYPE_BF16, AF_DTYPE_F32, AfEpilogue

_gn_ws = {}


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _p(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _chk(t: torch.Tensor, dtype, name: str) -> None:
    if not t.is_cuda:
        raise ValueError(f"{name}: expected a CUDA tensor (there is no CPU path)")
    if t.dtype != dtype:
        raise ValueError(f"{name}: expected {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name}: must be contiguous")


def _epilogue(out: torch.Tensor, bias=None, rowbias=None, rows_per_group=0, residual=None, geglu=False,
              ldo: int = 0, ldr: int = 0, gn_stats: Optional[torch.Tensor] = None, act: int = 0) -> AfEpilogue:
    # rowbias may be a column slice of a wider [groups, total] matrix: its row stride is passed along
    ep = AfEpilogue()
    if bias is not None:
        _chk(bias, torch.float32, "bias")
    if rowbias is not None:
        if rowbias.dtype != torch.float32 or not rowbias.is_cuda or rowbias.stride(-1) != 1:
            raise ValueError("rowbias must be a CUDA fp32 tensor with unit column stride")
    if residual is not None:
        _chk(residual, torch.float32, "residual")
    ep.bias = _p(bias)
    ep.rowbias = _p(rowbias)
    ep.rows_per_group = int(rows_per_group)
    ep.ld_rowbias = int(rowbias.stride(0)) if rowbias is not None and rowbias.dim() == 2 else 0
    ep.residual = _p(residual)
    ep.ldr = int(ldr)
    ep.out = out.data_ptr()
    ep.ldo = int(ldo)
    if out.dtype == torch.bfloat16:
        ep.out_dtype = AF_DTYPE_BF16
    elif out.dtype == torch.float32:
        ep.out_dtype = AF_DTYPE_F32
    else:
        raise ValueError(f"out dtype {out.dtype} unsupported")
    ep.geglu = 1 if geglu else 0
    ep.act = int(act)
    if gn_stats is not None:
        _chk(gn_stats, torch.float32, "gn_stats")
    ep.gn_stats = _p(gn_stats)
    ep.pair_mode = LAUNCH_OPTIONS.pair_mode
    ep.trace = _p(LAUNCH_OPTIONS.trace)
    ep.split_k = LAUNCH_OPTIONS.split_k
    if not geglu and LAUNCH_OPTIONS.split_k != 1:
        ws = _splitk_workspace(out.device)
        if ws is not None:
            ep.splitk_ws, ep.splitk_ws_bytes = ws.data_ptr(), ws.numel() * 4
    return ep


SPLITK_WS_BYTES = 16384 + 48 * (1 << 20)     # flag region + 48 MB of fp32 partial tiles
_splitk_ws = {}


def _splitk_workspace(device) -> Optional[torch.Tensor]:
    """Split-K workspace (af_epilogue.splitk_ws), or None for the whole-tile schedule.

    A split tile's finisher block spins until the blocks holding the other K ranges of the tile have run, which is only
    safe while the kernel's blocks are not kept off the SMs by ANOTHER kernel that is itself waiting the same way.  So
    per device the schedule is enabled for ONE eager stream at a time (it moves to another stream only once everything
    submitted to the previous one has completed - every path of this package is single-stream) and for launches recorded
    into CUDA graphs (replays are stream-ordered; graphs of one device must not replay concurrently with each other or
    with eager GEMMs); a GEMM on any other stream gets the whole-tile schedule.  Each of the two has its own workspace,
    zeroed once - the kernel leaves the flag region zero.  Nothing is allocated while a capture is in progress: the
    eager warm-up that precedes every capture creates both."""
    capturing = torch.cuda.is_current_stream_capturing()
    if device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    st = _splitk_ws.get(device.index)
    if capturing:
        return st["graph"] if st is not None else None
    cur = torch.cuda.current_stream(device)
    if st is None:
        st = _splitk_ws[device.index] = {
            "stream": cur,
            "eager": torch.zeros(SPLITK_WS_BYTES // 4, dtype=torch.float32, device=device),
            "graph": torch.zeros(SPLITK_WS_BYTES // 4, dtype=torch.float32, device=device)}
    if st["stream"].cuda_stream != cur.cuda_stream:
        if not st["stream"].query():
            return None
        st["stream"] = cur
    return st["eager"]


class _LaunchOptions:
    """Per-call options of af_gemm_bf16 / af_conv3x3_bf16 that the host mirror leaves at their defaults; tests and the
    measurement scripts override them for a `with launch_options(...)` block.  The state lives HERE, in the Python
    caller - the library itself keeps none."""
    pair_mode = 0      # AF_PAIR_AUTO
    trace = None       # device int64 tensor: GEMM timeline probe
    split_k = 0        # 0 auto, 1 never, n > 1: cut the tiles of the last partial wave into n K ranges


LAUNCH_OPTIONS = _LaunchOptions()


class launch_options:
    def __init__(self, pair_mode: Optional[int] = None, trace: Optional[torch.Tensor] = None,
                 split_k: Optional[int] = None):
        self.new = (pair_mode, trace, split_k)

    def __enter__(self):
        self.old = (LAUNCH_OPTIONS.pair_mode, LAUNCH_OPTIONS.trace, LAUNCH_OPTIONS.split_k)
        if self.new[0] is not None:
            LAUNCH_OPTIONS.pair_mode = int(self.new[0])
        LAUNCH_OPTIONS.trace = self.new[1]
        if self.new[2] is not None:
            LAUNCH_OPTIONS.split_k = int(self.new[2])
        return self

    def __exit__(self, *exc):
        LAUNCH_OPTIONS.pair_mode, LAUNCH_OPTIONS.trace, LAUNCH_OPTIONS.split_k = self.old
        return False


def gemm(a0: torch.Tensor, wt: torch.Tensor, out: torch.Tensor, *, a1: Optional[torch.Tensor] = None,
         bias=None, rowbias=None, rows_per_group=0, residual=None, geglu=False, ldo: int = 0, ldr: int = 0,
         bn: int = 0, M: Optional[int] = None, lda0: Optional[int] = None, K0: Optional[int] = None,
         gn_stats: Optional[torch.Tensor] = None, act: int = 0) -> torch.Tensor:
    """out[M, N] = [a0 | a1] @ wt^T (+ fused epilogue).  act=1: quick_gelu on (acc + bias).  a*: bf16 [M, K*]; wt: bf16 [N, K0+K1].
    gn_stats: fp32 [ceil(M/128)*4, N, 2] per-32-row (sum, sumsq) of the written values (see gn_stats_for_rows)."""
    lib = _lib.load()
    _chk(wt, torch.bfloat16, "wt")
    if a0.dtype != torch.bfloat16 or not a0.is_cuda:
        raise ValueError("a0 must be a CUDA bf16 tensor")
    M = int(a0.shape[0]) if M is None else M
    K0 = int(a0.shape[-1]) if K0 is None else K0
    lda0 = int(a0.stride(0)) if lda0 is None else lda0
    K1, lda1 = 0, 0
    if a1 is not None:
        _chk(a1, torch.bfloat16, "a1")
        K1, lda1 = int(a1.shape[-1]), int(a1.stride(0))
    N = int(wt.shape[0])
    if int(wt.shape[1]) != K0 + K1:
        raise ValueError(f"wt K={wt.shape[1]} != K0+K1={K0 + K1}")
    ep = _epilogue(out, bias, rowbias, rows_per_group, residual, geglu, ldo, ldr, gn_stats, act)
    rc = lib.af_gemm_bf16(a0.data_ptr(), lda0, K0, _p(a1), lda1, K1, wt.data_ptr(), M, N, byref(ep), bn, _stream())
    _lib.check(rc, "af_gemm_bf16")
    return out


def conv3x3(x0: torch.Tensor, wt: torch.Tensor, out: torch.Tensor, *, x1: Optional[torch.Tensor] = None, stride=1,
            bias=None, rowbias=None, residual=None, bn: int = 0,
            gn_stats: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x*: bf16 NHWC [B,H,W,C*]; wt: bf16 [Cout, 3, 3, C0+C1]; out: [B,Ho,Wo,Cout] fp32|bf16."""
    lib = _lib.load()
    _chk(x0, torch.bfloat16, "x0")
    _chk(wt, torch.bfloat16, "wt")
    B, H, W, C0 = (int(s) for s in x0.shape)
    C1 = 0
    if x1 is not None:
        _chk(x1, torch.bfloat16, "x1")
        C1 = int(x1.shape[-1])
    Cout = int(wt.shape[0])
    if wt.numel() != Cout * 9 * (C0 + C1):
        raise ValueError("conv3x3 weight shape mismatch")
    ep = _epilogue(out, bias, rowbias, 0, residual, gn_stats=gn_stats)
    rc = lib.af_conv3x3_bf16(x0.data_ptr(), C0, _p(x1), C1, wt.data_ptr(), B, H, W, Cout, stride, byref(ep), bn,
                             _stream())
    _lib.check(rc, "af_conv3x3_bf16")
    return out


def conv3x3_down01(x: torch.Tensor, wt: torch.Tensor, out: torch.Tensor, *, bias=None, bn: int = 0,
                   gn_stats: Optional[torch.Tensor] = None) -> torch.Tensor:
    """conv3x3 stride 2 of F.pad(x, (0,1,0,1)) (VAE encoder Downsample).  x: bf16 NHWC [B,H,W,C] (H, W even);
    wt: bf16 [Cout, 3, 3, C]; out: [B,H/2,W/2,Cout] fp32|bf16."""
    lib = _lib.load()
    _chk(x, torch.bfloat16, "x")
    _chk(wt, torch.bfloat16, "wt")
    B, H, W, C = (int(s) for s in x.shape)
    Cout = int(wt.shape[0])
    if wt.numel() != Cout * 9 * C:
        raise ValueError("conv3x3_down01 weight shape mismatch")
    ep = _epilogue(out, bias, gn_stats=gn_stats)
    rc = lib.af_conv3x3_down01_bf16(x.data_ptr(), C, wt.data_ptr(), B, H, W, Cout, byref(ep), bn, _stream())
    _lib.check(rc, "af_conv3x3_down01_bf16")
    return out


def attention(q: torch.Tensor, k: torch.Tensor, vt: torch.Tensor, out: torch.Tensor, *, B: int, heads: int, Nq: int,
              Nk: int, d: int, ldq: int, ldk: int, ldvt: int, kv_stride: int,
              key_mask: Optional[torch.Tensor] = None) -> torch.Tensor:
    lib = _lib.load()
    for t, n in ((q, "q"), (k, "k"), (vt, "vt"), (out, "out")):
        if t.dtype != torch.bfloat16 or not t.is_cuda:
            raise ValueError(f"{n} must be a CUDA bf16 tensor")
    if key_mask is not None:
        _chk(key_mask, torch.uint8, "key_mask")
    rc = lib.af_attention_bf16(q.data_ptr(), ldq, k.data_ptr(), ldk, vt.data_ptr(), ldvt, kv_stride, _p(key_mask),
                               out.data_ptr(), B, heads, Nq, Nk, d, _stream())
    _lib.check(rc, "af_attention_bf16")
    return out


class GNStats:
    """Per-channel partial GroupNorm statistics of one fp32 NHWC tensor: buf fp32 [B, slots, C, 2]
    (include/adaface_b200.h, "Statistics format").  Produced by a GEMM / conv epilogue or by groupnorm_stats."""

    __slots__ = ("buf", "slots", "C")

    def __init__(self, buf: torch.Tensor, slots: int, C: int):
        self.buf, self.slots, self.C = buf, slots, C


def gn_stats_for_gemm(B: int, HW: int, C: int, device) -> Optional[GNStats]:
    """Statistics buffer a GEMM epilogue can fill for an output of B*HW rows (None: geometry unsupported)."""
    if HW % 32 != 0:
        return None
    rows32 = (B * HW + 127) // 128 * 4
    return GNStats(torch.empty(rows32 * C * 2, dtype=torch.float32, device=device), HW // 32, C)


def gn_stats_for_conv(B: int, Ho: int, Wo: int, C: int, device) -> Optional[GNStats]:
    slots = _lib.load().af_conv3x3_gn_slots(Ho, Wo)
    if slots <= 0:
        return None
    return GNStats(torch.empty(B * slots * C * 2, dtype=torch.float32, device=device), slots, C)


def groupnorm_stats(x: torch.Tensor) -> GNStats:
    """Stand-alone statistics pass for a tensor no tensor-core kernel produced."""
    lib = _lib.load()
    _chk(x, torch.float32, "x")
    B, C = int(x.shape[0]), int(x.shape[-1])
    HW = x.numel() // (B * C)
    slots = lib.af_groupnorm_stats_slots(B, HW)
    st = GNStats(torch.empty(B * slots * C * 2, dtype=torch.float32, device=x.device), slots, C)
    rc = lib.af_groupnorm_stats(x.data_ptr(), C, B, HW, st.buf.data_ptr(), slots, _stream())
    _lib.check(rc, "af_groupnorm_stats")
    return st


def groupnorm_apply(x0: torch.Tensor, st0: GNStats, gamma: torch.Tensor, beta: torch.Tensor, eps: float, silu: bool,
                    out: torch.Tensor, *, x1: Optional[torch.Tensor] = None, st1: Optional[GNStats] = None,
                    raw: Optional[torch.Tensor] = None) -> torch.Tensor:
    """GroupNorm(32) [+SiLU] of [x0 | x1] from precomputed statistics: finalize (tiny) + ONE pass over the data."""
    lib = _lib.load()
    _chk(x0, torch.float32, "x0")
    _chk(out, torch.bfloat16, "out")
    B, C0 = int(x0.shape[0]), int(x0.shape[-1])
    HW = x0.numel() // (B * C0)
    C1 = 0
    if x1 is not None:
        _chk(x1, torch.float32, "x1")
        C1 = int(x1.shape[-1])
        if st1 is None or st1.C != C1:
            raise ValueError("groupnorm_apply: x1 needs matching statistics")
    if st0.C != C0:
        raise ValueError("groupnorm_apply: statistics / tensor channel mismatch")
    if raw is not None:
        _chk(raw, torch.bfloat16, "raw")
    mr = torch.empty(B * 64, dtype=torch.float32, device=x0.device)
    rc = lib.af_groupnorm_finalize(st0.buf.data_ptr(), C0, st0.slots, st1.buf.data_ptr() if C1 else None, C1,
                                   st1.slots if C1 else 0, B, HW, float(eps), mr.data_ptr(), _stream())
    _lib.check(rc, "af_groupnorm_finalize")
    rc = lib.af_groupnorm_apply(x0.data_ptr(), C0, _p(x1), C1, B, HW, mr.data_ptr(), gamma.data_ptr(), beta.data_ptr(),
                                1 if silu else 0, out.data_ptr(), _p(raw), _stream())
    _lib.check(rc, "af_groupnorm_apply")
    return out


def _gn_workspace(B: int, C: int, device) -> torch.Tensor:
    key = (B, C, device)
    ws = _gn_ws.get(key)
    if ws is None:
        n = _lib.load().af_groupnorm_workspace_bytes(B, C)
        ws = torch.empty(n // 4, dtype=torch.float32, device=device)
        _gn_ws[key] = ws
    return ws


def groupnorm_silu(x0: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float, silu: bool,
                   out: torch.Tensor, *, x1: Optional[torch.Tensor] = None, raw: Optional[torch.Tensor] = None,
                   workspace: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x*: fp32 NHWC [B, H, W, C*] (or [B, HW, C*]); out: bf16 [B, HW, C0+C1].  All-in-one (statistics passes
    included); the UNet fast path uses groupnorm_apply with producer-side statistics instead."""
    lib = _lib.load()
    _chk(x0, torch.float32, "x0")
    _chk(out, torch.bfloat16, "out")
    B, C0 = int(x0.shape[0]), int(x0.shape[-1])
    HW = x0.numel() // (B * C0)
    C1 = 0
    if x1 is not None:
        _chk(x1, torch.float32, "x1")
        C1 = int(x1.shape[-1])
    if raw is not None:
        _chk(raw, torch.bfloat16, "raw")
    ws = workspace if workspace is not None else _gn_workspace(B, C0 + C1, x0.device)
    rc = lib.af_groupnorm_silu(x0.data_ptr(), C0, _p(x1), C1, B, HW, gamma.data_ptr(), beta.data_ptr(), float(eps),
                               1 if silu else 0, out.data_ptr(), _p(raw), ws.data_ptr(), _stream())
    _lib.check(rc, "af_groupnorm_silu")
    return out


def layernorm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float, out: torch.Tensor) -> torch.Tensor:
    """out bf16 (GEMM operand) or fp32 (CLIP final_layer_norm)."""
    lib = _lib.load()
    _chk(x, torch.float32, "x")
    C = int(x.shape[-1])
    if out.dtype == torch.float32:
        _chk(out, torch.float32, "out")
        rc = lib.af_layernorm_f32(x.data_ptr(), x.numel() // C, C, gamma.data_ptr(), beta.data_ptr(), float(eps),
                                  out.data_ptr(), _stream())
        _lib.check(rc, "af_layernorm_f32")
        return out
    _chk(out, torch.bfloat16, "out")
    rc = lib.af_layernorm(x.data_ptr(), x.numel() // C, C, gamma.data_ptr(), beta.data_ptr(), float(eps),
                          out.data_ptr(), _stream())
    _lib.check(rc, "af_layernorm")
    return out


def conv_in(x_nchw: torch.Tensor, w: torch.Tensor, bias: torch.Tensor, out_nhwc: torch.Tensor) -> torch.Tensor:
    lib = _lib.load()
    _chk(x_nchw, torch.float32, "x")
    _chk(w, torch.float32, "w")
    _chk(out_nhwc, torch.float32, "out")
    B, Cin, H, W = (int(s) for s in x_nchw.shape)
    rc = lib.af_conv_in(x_nchw.data_ptr(), w.data_ptr(), _p(bias), out_nhwc.data_ptr(), B, Cin, H, W, int(w.shape[0]),
                        _stream())
    _lib.check(rc, "af_conv_in")
    return out_nhwc


def conv_out(x_nhwc: torch.Tensor, w_packed: torch.Tensor, bias: torch.Tensor, out_nchw: torch.Tensor) -> torch.Tensor:
    lib = _lib.load()
    _chk(x_nhwc, torch.bfloat16, "x")
    _chk(w_packed, torch.float32, "w")
    _chk(out_nchw, torch.float32, "out")
    B, H, W, C = (int(s) for s in x_nhwc.shape)
    rc = lib.af_conv_out(x_nhwc.data_ptr(), w_packed.data_ptr(), _p(bias), out_nchw.data_ptr(), B, H, W, C,
                         int(w_packed.shape[0]), _stream())
    _lib.check(rc, "af_conv_out")
    return out_nchw


def nhwc_to_nchw(x_nhwc: torch.Tensor, out_nchw: torch.Tensor) -> torch.Tensor:
    """x fp32 [B,H,W,Cp] -> out fp32 [B,Cout,H,W] (first Cout <= 4 channels)."""
    lib = _lib.load()
    _chk(x_nhwc, torch.float32, "x")
    _chk(out_nchw, torch.float32, "out")
    B, H, W, Cp = (int(v) for v in x_nhwc.shape)
    rc = lib.af_nhwc_to_nchw(x_nhwc.data_ptr(), out_nchw.data_ptr(), B, H * W, Cp, int(out_nchw.shape[1]), _stream())
    _lib.check(rc, "af_nhwc_to_nchw")
    return out_nchw


def timestep_embedding(t: torch.Tensor, dim: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    lib = _lib.load()
    _chk(t, torch.float32, "t")
    B = int(t.shape[0])
    if out is None:
        out = torch.empty(B, dim, dtype=torch.float32, device=t.device)
    rc = lib.af_timestep_embedding(t.data_ptr(), out.data_ptr(), B, dim, _stream())
    _lib.check(rc, "af_timestep_embedding")
    return out


def linear_small(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], out: torch.Tensor, *,
                 silu_in=False, silu_out=False) -> torch.Tensor:
    lib = _lib.load()
    _chk(x, torch.float32, "x")
    _chk(w, torch.float32, "w")
    _chk(out, torch.float32, "out")
    M, K = int(x.shape[0]), int(x.shape[1])
    N = int(w.shape[0])
    rc = lib.af_linear_small(x.data_ptr(), w.data_ptr(), _p(bias), out.data_ptr(), M, N, K, int(silu_in),
                             int(silu_out), _stream())
    _lib.check(rc, "af_linear_small")
    return out


def cast_bf16(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    lib = _lib.load()
    _chk(x, torch.float32, "x")
    if out is None:
        out = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
    rc = lib.af_cast_bf16(x.data_ptr(), out.data_ptr(), x.numel(), _stream())
    _lib.check(rc, "af_cast_bf16")
    return out


def channel_mix4(x_nchw: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], in_scale: float = 1.0) -> torch.Tensor:
    """1x1 conv over <= 4 channels of an NCHW fp32 tensor with an input scale (VAE post_quant_conv on z / scale_factor)."""
    lib = _lib.load()
    _chk(x_nchw, torch.float32, "x")
    _chk(w, torch.float32, "w")
    B, Cin, H, W = (int(s) for s in x_nchw.shape)
    Cout = int(w.shape[0])
    out = torch.empty(B, Cout, H, W, dtype=torch.float32, device=x_nchw.device)
    rc = lib.af_channel_mix4(x_nchw.data_ptr(), w.data_ptr(), _p(bias), float(in_scale), B, Cin, Cout, H * W,
                             out.data_ptr(), _stream())
    _lib.check(rc, "af_channel_mix4")
    return out


def vae_posterior(moments_nhwc: torch.Tensor, noise: Optional[torch.Tensor], out_scale: float, z: torch.Tensor,
                  mean: Optional[torch.Tensor] = None, logvar: Optional[torch.Tensor] = None) -> torch.Tensor:
    """DiagonalGaussianDistribution of the encoder moments fp32 NHWC [B,H,W,2*zc]: z = out_scale * (mean + std * noise)
    (noise None: out_scale * mean), and optionally mean / clamped logvar; z, noise, mean, logvar fp32 NCHW [B,zc,H,W]."""
    lib = _lib.load()
    _chk(moments_nhwc, torch.float32, "moments")
    _chk(z, torch.float32, "z")
    B, H, W, C2 = (int(s) for s in moments_nhwc.shape)
    zc = C2 // 2
    shape = (B, zc, H, W)
    for t, n in ((noise, "noise"), (z, "z"), (mean, "mean"), (logvar, "logvar")):
        if t is not None:
            _chk(t, torch.float32, n)
            if tuple(t.shape) != shape:
                raise ValueError(f"vae_posterior: {n} shape {tuple(t.shape)} != {shape}")
    rc = lib.af_vae_posterior(moments_nhwc.data_ptr(), B, H * W, zc, _p(noise), float(out_scale), z.data_ptr(), _p(mean),
                              _p(logvar), _stream())
    _lib.check(rc, "af_vae_posterior")
    return z


def softmax_rows(x: torch.Tensor, scale: float, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out[r] = softmax(scale * x[r]) per row: fp32 [rows, n] -> bf16 [rows, n] (VAE AttnBlock, model.py:188-193)."""
    lib = _lib.load()
    _chk(x, torch.float32, "x")
    rows, n = (int(s) for s in x.shape)
    if out is None:
        out = torch.empty(rows, n, dtype=torch.bfloat16, device=x.device)
    _chk(out, torch.bfloat16, "out")
    rc = lib.af_softmax_rows(x.data_ptr(), int(x.stride(0)), rows, n, float(scale), out.data_ptr(), int(out.stride(0)),
                             _stream())
    _lib.check(rc, "af_softmax_rows")
    return out


def upsample2x_cast(x_nhwc: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    lib = _lib.load()
    _chk(x_nhwc, torch.float32, "x")
    _chk(out, torch.bfloat16, "out")
    B, H, W, C = (int(s) for s in x_nhwc.shape)
    rc = lib.af_upsample2x_cast(x_nhwc.data_ptr(), out.data_ptr(), B, H, W, C, _stream())
    _lib.check(rc, "af_upsample2x_cast")
    return out


def cfg_ddim_update(x: torch.Tensor, eps: torch.Tensor, coef_table: torch.Tensor, x_prev: torch.Tensor,
                    pred_x0: Optional[torch.Tensor], *, has_uncond: bool, noise: Optional[torch.Tensor] = None,
                    step_idx: Optional[torch.Tensor] = None) -> torch.Tensor:
    lib = _lib.load()
    _chk(x, torch.float32, "x")
    _chk(eps, torch.float32, "eps")
    _chk(coef_table, torch.float32, "coef_table")
    rc = lib.af_cfg_ddim_update(x.data_ptr(), eps.data_ptr(), int(has_uncond), _p(noise), coef_table.data_ptr(),
                                _p(step_idx), x_prev.data_ptr(), _p(pred_x0), x.numel(), _stream())
    _lib.check(rc, "af_cfg_ddim_update")
    return x_prev


def advance_step(step_idx: torch.Tensor, t_table: torch.Tensor, t_buf: torch.Tensor, num_steps: int) -> None:
    lib = _lib.load()
    rc = lib.af_advance_step(step_idx.data_ptr(), t_table.data_ptr(), t_buf.data_ptr(), int(t_buf.shape[0]),
                             int(num_steps), _stream())
    _lib.check(rc, "af_advance_step")


# ---------------------------------------------------------------------------------------------------
# conditioning path (text.cu)
# ---------------------------------------------------------------------------------------------------
def attention_small(qkv: torch.Tensor, out: torch.Tensor, *, B: int, heads: int, L: int, k_off: int, v_off: int,
                    mult: int = 1, scale: float = 0.125, causal: bool = True) -> torch.Tensor:
    """qkv bf16 [B*L, ldq] (q | k | v column blocks, keys/values [head][r][64] for MKV) -> out bf16 [B*L, heads*64]."""
    lib = _lib.load()
    _chk(qkv, torch.bfloat16, "qkv")
    _chk(out, torch.bfloat16, "out")
    rc = lib.af_attention_small(qkv.data_ptr(), int(qkv.stride(0)), int(k_off), int(v_off), out.data_ptr(),
                                int(out.stride(0)), B, heads, L, mult, float(scale), int(causal), _stream())
    _lib.check(rc, "af_attention_small")
    return out


def gather_rows(table: torch.Tensor, ids: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out[..., :] = table[ids[...], :] (fp32, exact copies)."""
    lib = _lib.load()
    _chk(table, torch.float32, "table")
    _chk(ids, torch.int64, "ids")
    if out is None:
        out = torch.empty(*ids.shape, table.shape[1], dtype=torch.float32, device=table.device)
    rc = lib.af_gather_rows(table.data_ptr(), ids.data_ptr(), out.data_ptr(), ids.numel(), int(table.shape[1]),
                            int(table.shape[0]), _stream())
    _lib.check(rc, "af_gather_rows")
    return out


def add_pos(x: torch.Tensor, pos: torch.Tensor) -> torch.Tensor:
    """x [B, L, D] += pos[:L] in place."""
    lib = _lib.load()
    _chk(x, torch.float32, "x")
    _chk(pos, torch.float32, "pos")
    L, D = int(x.shape[-2]), int(x.shape[-1])
    rc = lib.af_add_pos(x.data_ptr(), pos.data_ptr(), x.numel() // D, L, D, _stream())
    _lib.check(rc, "af_add_pos")
    return x


def find_first_token(ids: torch.Tensor, token: int) -> torch.Tensor:
    """ids int64 [R, L] -> int32 [R]: first position of `token` per row or -1."""
    lib = _lib.load()
    _chk(ids, torch.int64, "ids")
    R, L = int(ids.shape[0]), int(ids.shape[1])
    out = torch.empty(R, dtype=torch.int32, device=ids.device)
    rc = lib.af_find_first_token(ids.data_ptr(), R, L, int(token), out.data_ptr(), _stream())
    _lib.check(rc, "af_find_first_token")
    return out


def splice_rows(dst: torch.Tensor, src: torch.Tensor, start: torch.Tensor, src_index: Optional[torch.Tensor] = None
                ) -> torch.Tensor:
    """dst fp32 [R, L, D]; src fp32 [S, K, D]; start int32 [R] (-1: untouched); src_index int32 [R] or None."""
    lib = _lib.load()
    _chk(dst, torch.float32, "dst")
    _chk(src, torch.float32, "src")
    _chk(start, torch.int32, "start")
    if src_index is not None:
        _chk(src_index, torch.int32, "src_index")
    R, L, D = (int(v) for v in dst.shape)
    rc = lib.af_splice_rows(dst.data_ptr(), src.data_ptr(), start.data_ptr(), _p(src_index), R, L, int(src.shape[1]), D,
                            _stream())
    _lib.check(rc, "af_splice_rows")
    return dst


def weighted_sum(a: torch.Tensor, b: torch.Tensor, c: Optional[torch.Tensor], w, out: Optional[torch.Tensor] = None
                 ) -> torch.Tensor:
    """out = w[0]*a + w[1]*b (+ w[2]*c), fp32."""
    lib = _lib.load()
    for t in (a, b) + ((c,) if c is not None else ()):
        _chk(t, torch.float32, "operand")
    if out is None:
        out = torch.empty_like(a)
    rc = lib.af_weighted_sum(a.data_ptr(), b.data_ptr(), _p(c), float(w[0]), float(w[1]), float(w[2]) if c is not None else 0.0,
                             out.data_ptr(), a.numel(), _stream())
    _lib.check(rc, "af_weighted_sum")
    return out


# ---------------------------------------------------------------------------------------------------
# training step: backward kernels (train.cu, bgemm.cu)
# ---------------------------------------------------------------------------------------------------
def attention_lse(q, k, vt, out, lse, *, B, heads, Nq, Nk, d, ldq, ldk, ldvt, kv_stride, key_mask=None):
    """af_attention_bf16 that also writes lse fp32 [B, heads, Nq] (log2-sum-exp of each query row)."""
    lib = _lib.load()
    _chk(lse, torch.float32, "lse")
    if key_mask is not None:
        _chk(key_mask, torch.uint8, "key_mask")
    rc = lib.af_attention_bf16_lse(q.data_ptr(), ldq, k.data_ptr(), ldk, vt.data_ptr(), ldvt, kv_stride, _p(key_mask),
                                   out.data_ptr(), lse.data_ptr(), B, heads, Nq, Nk, d, _stream())
    _lib.check(rc, "af_attention_bf16_lse")
    return out


def check_key_mask(key_mask: torch.Tensor, B: int, N: int, name: str = "key_mask") -> None:
    """A self-attention key mask as the masked backward kernels read it: uint8 [B, N] (1 = attend), contiguous, CUDA."""
    if not isinstance(key_mask, torch.Tensor):
        raise ValueError(f"{name}: expected a torch.Tensor, got {type(key_mask).__name__}")
    if key_mask.dtype != torch.uint8:
        raise ValueError(f"{name}: expected torch.uint8, got {key_mask.dtype}")
    if tuple(key_mask.shape) != (B, N):
        raise ValueError(f"{name}: expected shape {(B, N)}, got {tuple(key_mask.shape)}")
    if not key_mask.is_contiguous():
        raise ValueError(f"{name}: must be contiguous")
    if not key_mask.is_cuda:
        raise ValueError(f"{name}: expected a CUDA tensor (there is no CPU path)")
    if key_mask.data_ptr() % 16:
        raise ValueError(f"{name}: must start on a 16-byte boundary")


def bgemm(A, lda, sA, Bm, ldb, sB, C, ldc, sC, *, M, N, K, nb0, nb1, mode=0, vec=None, sV=(0, 0), P=None, ldp=0,
          sP=(0, 0), valid_rows=0, valid_cols=0, alpha=1.0, key_mask=None):
    """Batched strided C[z] = epi(A[z] . B[z]^T); A/B/C/P are (tensor, element offset) pairs or tensors.
    key_mask: uint8 [nb0, keys] self-attention key mask (modes 1-4, af_bgemm_masked_bf16), keys = valid_cols of modes
    1 / 3, valid_rows of modes 2 / 4; the same mask serves every head (z = (sample, head))."""
    if key_mask is not None:
        if mode not in (1, 2, 3, 4):
            raise ValueError(f"bgemm: mode {mode} takes no key mask")
        nk = (valid_cols or N) if mode in (1, 3) else (valid_rows or M)
        check_key_mask(key_mask, nb0, nk)
    lib = _lib.load()

    def ptr(t):
        if isinstance(t, tuple):
            return t[0].data_ptr() + t[1] * t[0].element_size()
        return t.data_ptr()

    Ct = C[0] if isinstance(C, tuple) else C
    g = _lib.AfBgemm()
    g.A, g.lda, g.sA0, g.sA1 = ptr(A), lda, sA[0], sA[1]
    g.B, g.ldb, g.sB0, g.sB1 = ptr(Bm), ldb, sB[0], sB[1]
    g.C, g.ldc, g.sC0, g.sC1 = ptr(C), ldc, sC[0], sC[1]
    g.c_dtype = AF_DTYPE_F32 if Ct.dtype == torch.float32 else AF_DTYPE_BF16
    g.vec, g.sV0, g.sV1 = (vec.data_ptr() if vec is not None else None), sV[0], sV[1]
    g.P, g.ldp, g.sP0, g.sP1 = (ptr(P) if P is not None else None), ldp, sP[0], sP[1]
    g.M, g.N, g.K, g.nb0, g.nb1, g.mode = M, N, K, nb0, nb1, mode
    g.valid_rows, g.valid_cols, g.alpha = valid_rows, valid_cols, float(alpha)
    if key_mask is None:
        rc = lib.af_bgemm_bf16(byref(g), _stream())
        _lib.check(rc, "af_bgemm_bf16")
        return
    rc = lib.af_bgemm_masked_bf16(byref(g), key_mask.data_ptr(), int(key_mask.shape[1]), 0, _stream())
    _lib.check(rc, "af_bgemm_masked_bf16")


def groupnorm_mean_rstd(x: torch.Tensor, st: GNStats, eps: float) -> torch.Tensor:
    """mean / rstd [B, 32, 2] of a single-source GroupNorm from its partial statistics."""
    lib = _lib.load()
    B, C = int(x.shape[0]), int(x.shape[-1])
    HW = x.numel() // (B * C)
    mr = torch.empty(B * 64, dtype=torch.float32, device=x.device)
    rc = lib.af_groupnorm_finalize(st.buf.data_ptr(), C, st.slots, None, 0, 0, B, HW, float(eps), mr.data_ptr(), _stream())
    _lib.check(rc, "af_groupnorm_finalize")
    return mr


def groupnorm_apply_mr(x: torch.Tensor, mr: torch.Tensor, gamma, beta, silu: bool, out: torch.Tensor) -> torch.Tensor:
    lib = _lib.load()
    B, C = int(x.shape[0]), int(x.shape[-1])
    HW = x.numel() // (B * C)
    rc = lib.af_groupnorm_apply(x.data_ptr(), C, None, 0, B, HW, mr.data_ptr(), gamma.data_ptr(), beta.data_ptr(),
                                1 if silu else 0, out.data_ptr(), None, _stream())
    _lib.check(rc, "af_groupnorm_apply")
    return out


def groupnorm_bwd(x, mr, gamma, beta, silu: bool, dy: torch.Tensor, dres: Optional[torch.Tensor] = None) -> torch.Tensor:
    lib = _lib.load()
    _chk(x, torch.float32, "x")
    _chk(dy, torch.bfloat16, "dy")
    if dres is not None:
        _chk(dres, torch.float32, "dres")
    B, C = int(x.shape[0]), int(x.shape[-1])
    HW = x.numel() // (B * C)
    ws = torch.empty(lib.af_groupnorm_bwd_workspace_floats(B, C, HW), dtype=torch.float32, device=x.device)
    dx = torch.empty_like(x)
    rc = lib.af_groupnorm_bwd(x.data_ptr(), C, B, HW, mr.data_ptr(), gamma.data_ptr(), beta.data_ptr(), int(silu),
                              dy.data_ptr(), _p(dres), dx.data_ptr(), ws.data_ptr(), _stream())
    _lib.check(rc, "af_groupnorm_bwd")
    return dx


def layernorm_bwd(x, gamma, eps, dy, dres=None, dgamma=None, dbeta=None) -> torch.Tensor:
    lib = _lib.load()
    _chk(x, torch.float32, "x")
    if not dy.is_contiguous() or dy.dtype not in (torch.float32, torch.bfloat16):
        raise ValueError("dy must be contiguous fp32 / bf16")
    C = int(x.shape[-1])
    dx = torch.empty_like(x)
    rc = lib.af_layernorm_bwd(x.data_ptr(), x.numel() // C, C, gamma.data_ptr(), float(eps), dy.data_ptr(),
                              AF_DTYPE_F32 if dy.dtype == torch.float32 else AF_DTYPE_BF16, _p(dres), dx.data_ptr(),
                              _p(dgamma), _p(dbeta), _stream())
    _lib.check(rc, "af_layernorm_bwd")
    return dx


def geglu_fwd(proj: torch.Tensor) -> torch.Tensor:
    lib = _lib.load()
    _chk(proj, torch.bfloat16, "proj")
    T, F2 = int(proj.shape[0]), int(proj.shape[1])
    h = torch.empty(T, F2 // 2, dtype=torch.bfloat16, device=proj.device)
    _lib.check(lib.af_geglu_fwd(proj.data_ptr(), T, F2 // 2, h.data_ptr(), _stream()), "af_geglu_fwd")
    return h


def geglu_bwd(proj: torch.Tensor, dh: torch.Tensor) -> torch.Tensor:
    lib = _lib.load()
    _chk(proj, torch.bfloat16, "proj")
    _chk(dh, torch.bfloat16, "dh")
    T, F2 = int(proj.shape[0]), int(proj.shape[1])
    dproj = torch.empty_like(proj)
    _lib.check(lib.af_geglu_bwd(proj.data_ptr(), dh.data_ptr(), T, F2 // 2, dproj.data_ptr(), _stream()), "af_geglu_bwd")
    return dproj


def quick_gelu(x: torch.Tensor, dy: Optional[torch.Tensor] = None) -> torch.Tensor:
    lib = _lib.load()
    _chk(x, torch.bfloat16, "x")
    if dy is not None:
        _chk(dy, torch.bfloat16, "dy")
    out = torch.empty_like(x)
    _lib.check(lib.af_quick_gelu(x.data_ptr(), _p(dy), x.numel(), out.data_ptr(), _stream()), "af_quick_gelu")
    return out


def xattn_explicit(q, k, vt, *, B, heads, N, nk, d, ldq, ldk, ldvt, kv_stride, override=None, ov_cols=None,
                   want_out=True, want_scores=False, want_attn=False, want_q=False):
    """Materialised-score cross-attention (af_xattn_explicit).  -> dict(out, attnscore, attn, q) of the requested parts."""
    lib = _lib.load()
    dev = q.device
    r = {"out": torch.empty(B * N, heads * d, dtype=torch.bfloat16, device=dev) if want_out else None,
         "attnscore": torch.empty(B, heads, N, nk, dtype=torch.float32, device=dev) if want_scores else None,
         "attn": torch.empty(B, heads, N, nk, dtype=torch.float32, device=dev) if want_attn else None,
         "q": torch.empty(B, heads, N, d, dtype=torch.float32, device=dev) if want_q else None}
    n_ov = int(ov_cols.shape[1]) if ov_cols is not None else 0
    rc = lib.af_xattn_explicit(q.data_ptr(), ldq, k.data_ptr(), ldk, vt.data_ptr(), ldvt, kv_stride, _p(override),
                               _p(ov_cols), n_ov, _p(r["out"]), _p(r["attn"]), _p(r["attnscore"]), _p(r["q"]), B, heads, N,
                               nk, d, _stream())
    _lib.check(rc, "af_xattn_explicit")
    return r


def conv_attn_scores(score, cols, *, B, heads, Hf, Wf, nk, ks):
    lib = _lib.load()
    ov = torch.empty(B, heads, Hf * Wf, ks * ks, dtype=torch.float32, device=score.device)
    rc = lib.af_conv_attn_scores(score.data_ptr(), cols.data_ptr(), B, heads, Hf, Wf, nk, ks, ov.data_ptr(), _stream())
    _lib.check(rc, "af_conv_attn_scores")
    return ov


def attention_bwd(q, k, vp, dop, qT, kT, dOT, lse, delta, *, B, heads, N, d, key_mask=None):
    """dQ [B*N, h*dp], dK [B*N, h*dp], dV [B*N, h*d] (bf16) of the long self-attention (af_attention_bwd_bf16).
    key_mask: uint8 [B, N] self-attention key mask (af_attention_bwd_masked_bf16)."""
    if key_mask is not None:
        check_key_mask(key_mask, B, N)
    lib = _lib.load()
    dp = 48 if d == 40 else d
    dev = q.device
    dq = torch.empty(B * N, heads * dp, dtype=torch.bfloat16, device=dev)
    dk = torch.empty(B * N, heads * dp, dtype=torch.bfloat16, device=dev)
    dv = torch.empty(B * N, heads * d, dtype=torch.bfloat16, device=dev)
    for t in (q, k, vp, dop, qT, kT, dOT):
        if t.dtype != torch.bfloat16 or t.stride(-1) != 1:
            raise ValueError("attention_bwd: bf16 row-major operands expected")
    if key_mask is None:
        rc = lib.af_attention_bwd_bf16(q.data_ptr(), int(q.stride(0)), k.data_ptr(), int(k.stride(0)), vp.data_ptr(),
                                       int(vp.stride(0)), dop.data_ptr(), int(dop.stride(0)), qT.data_ptr(),
                                       int(qT.stride(0)), kT.data_ptr(), int(kT.stride(0)), dOT.data_ptr(),
                                       int(dOT.stride(0)), lse.data_ptr(), delta.data_ptr(), dq.data_ptr(), heads * dp,
                                       dk.data_ptr(), heads * dp, dv.data_ptr(), heads * d, B, heads, N, d, _stream())
        _lib.check(rc, "af_attention_bwd_bf16")
        return dq, dk, dv
    rc = lib.af_attention_bwd_masked_bf16(q.data_ptr(), int(q.stride(0)), k.data_ptr(), int(k.stride(0)), vp.data_ptr(),
                                          int(vp.stride(0)), dop.data_ptr(), int(dop.stride(0)), qT.data_ptr(),
                                          int(qT.stride(0)), kT.data_ptr(), int(kT.stride(0)), dOT.data_ptr(),
                                          int(dOT.stride(0)), lse.data_ptr(), delta.data_ptr(), key_mask.data_ptr(),
                                          dq.data_ptr(), heads * dp, dk.data_ptr(), heads * dp, dv.data_ptr(), heads * d,
                                          B, heads, N, d, _stream())
    _lib.check(rc, "af_attention_bwd_masked_bf16")
    return dq, dk, dv


def rowdot_heads(a: torch.Tensor, b: torch.Tensor, B: int, N: int, heads: int, d: int) -> torch.Tensor:
    lib = _lib.load()
    _chk(a, torch.bfloat16, "a")
    _chk(b, torch.bfloat16, "b")
    delta = torch.empty(B, heads, N, dtype=torch.float32, device=a.device)
    _lib.check(lib.af_rowdot_heads(a.data_ptr(), b.data_ptr(), B, N, heads, d, delta.data_ptr(), _stream()), "af_rowdot_heads")
    return delta


def attention_small_bwd(qkv, dout, *, B, heads, L, k_off, v_off, mult=1, scale=0.125, causal=True) -> torch.Tensor:
    lib = _lib.load()
    _chk(qkv, torch.bfloat16, "qkv")
    _chk(dout, torch.bfloat16, "dout")
    dqkv = torch.zeros_like(qkv)
    rc = lib.af_attention_small_bwd(qkv.data_ptr(), int(qkv.stride(0)), int(k_off), int(v_off), dout.data_ptr(),
                                    int(dout.stride(0)), dqkv.data_ptr(), B, heads, L, mult, float(scale), int(causal),
                                    _stream())
    _lib.check(rc, "af_attention_small_bwd")
    return dqkv


def conv_out_dgrad(dout_nchw: torch.Tensor, w: torch.Tensor, C: int) -> torch.Tensor:
    lib = _lib.load()
    _chk(dout_nchw, torch.float32, "dout")
    _chk(w, torch.float32, "w")
    B, Cout, H, W = (int(v) for v in dout_nchw.shape)
    dy = torch.empty(B, H, W, C, dtype=torch.bfloat16, device=dout_nchw.device)
    _lib.check(lib.af_conv_out_dgrad(dout_nchw.data_ptr(), w.data_ptr(), B, H, W, C, Cout, dy.data_ptr(), _stream()),
               "af_conv_out_dgrad")
    return dy


def sumpool2x2(x: torch.Tensor) -> torch.Tensor:
    lib = _lib.load()
    _chk(x, torch.float32, "x")
    B, H2, W2, C = (int(v) for v in x.shape)
    out = torch.empty(B, H2 // 2, W2 // 2, C, dtype=torch.float32, device=x.device)
    _lib.check(lib.af_sumpool2x2(x.data_ptr(), B, H2 // 2, W2 // 2, C, out.data_ptr(), _stream()), "af_sumpool2x2")
    return out


def zero_insert2x(x: torch.Tensor) -> torch.Tensor:
    lib = _lib.load()
    _chk(x, torch.float32, "x")
    B, H, W, C = (int(v) for v in x.shape)
    out = torch.empty(B, 2 * H, 2 * W, C, dtype=torch.bfloat16, device=x.device)
    _lib.check(lib.af_zero_insert2x(x.data_ptr(), B, H, W, C, out.data_ptr(), _stream()), "af_zero_insert2x")
    return out


def transpose_to_bf16(x: torch.Tensor, ldo: Optional[int] = None) -> torch.Tensor:
    """x [R, C] fp32 | bf16 -> bf16 [C, ldo] (ldo = R rounded up to 8), zero padded."""
    lib = _lib.load()
    if x.dtype not in (torch.float32, torch.bfloat16) or not x.is_contiguous():
        raise ValueError("transpose_to_bf16: contiguous fp32 / bf16 expected")
    R, C = int(x.shape[0]), int(x.shape[1])
    ldo = (R + 7) // 8 * 8 if ldo is None else ldo
    out = torch.empty(C, ldo, dtype=torch.bfloat16, device=x.device)
    rc = lib.af_transpose_to_bf16(x.data_ptr(), AF_DTYPE_F32 if x.dtype == torch.float32 else AF_DTYPE_BF16, R, C, ldo,
                                  out.data_ptr(), _stream())
    _lib.check(rc, "af_transpose_to_bf16")
    return out
