"""CPU checks of the drop-in boundary: the C-ABI library loads without a GPU and exports every symbol
include/adaface_b200.h declares; the Python binding table mirrors the header; the host modules keep the
reference's state_dict key names; and the product path refuses to run without CUDA (no CPU fallback)."""
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "adaface_b200.h")


def _declared():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(af_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol(lib):
    names = _declared()
    assert len(names) >= 17
    for n in names:
        assert hasattr(lib._cdll, n), f"{n} declared in adaface_b200.h but not exported"


def test_binding_table_matches_header():
    from adaprompt_b200 import _lib
    assert sorted(_lib.SIGNATURES) == _declared()


def test_version_and_error_string(lib):
    assert lib.af_version() == 202
    assert isinstance(lib.af_last_error(), bytes)


def test_bad_arguments_are_rejected_without_a_gpu(lib):
    """Argument validation happens before any CUDA call: negative rc + message."""
    from ctypes import byref
    from adaprompt_b200._lib import AfEpilogue
    ep = AfEpilogue()
    rc = lib.af_gemm_bf16(None, 0, 0, None, 0, 0, None, 0, 0, byref(ep), 0, None)
    assert rc < 0 and b"null" in lib.af_last_error()
    rc = lib.af_attention_bf16(1, 8, 1, 8, 1, 8, 8, None, 1, 1, 8, 8, 8, 64, None)
    assert rc < 0 and b"head dim" in lib.af_last_error()
    rc = lib.af_layernorm(1, 4, 30, 1, 1, 1e-5, 1, None)
    assert rc < 0


def test_state_dict_keys_match_reference_names():
    from adaprompt_b200.ldm_lite import SD15_UNET_CONFIG
    from adaprompt_b200.unet import UNetModel
    from oracle.unet_oracle import UNetSpec
    with torch.device("meta"):
        m = UNetModel(**SD15_UNET_CONFIG)
    sd = m.state_dict()
    spec = UNetSpec().state_spec()   # pinned against the reference's own state_dict in oracle/make_golden.py
    assert list(sd.keys()) == list(spec.keys())
    assert all(tuple(sd[k].shape) == spec[k] for k in spec)
    assert sum(v.numel() for v in sd.values()) == 859_520_964   # SURVEY.md section 6: 859.52 M parameters
    for k in ("input_blocks.1.1.transformer_blocks.0.attn1.to_q.weight", "middle_block.1.proj_out.weight",
              "output_blocks.11.0.skip_connection.weight", "input_blocks.3.0.op.weight",
              "output_blocks.2.1.conv.weight", "time_embed.2.bias", "out.2.weight",
              "input_blocks.4.1.transformer_blocks.0.ff.net.0.proj.weight"):
        assert k in sd


def test_no_cpu_fallback():
    from adaprompt_b200.unet import ResBlock
    from adaprompt_b200 import ops
    rb = ResBlock(320, 1280, 0.0, out_channels=320)
    with pytest.raises(RuntimeError):
        rb(torch.randn(1, 320, 8, 8), torch.randn(1, 1280))
    with pytest.raises(ValueError):
        ops.cast_bf16(torch.randn(8))


def test_unsupported_configs_raise():
    from adaprompt_b200.unet import ResBlock, UNetModel
    with pytest.raises(NotImplementedError):
        ResBlock(320, 1280, 0.0, use_scale_shift_norm=True)
    with pytest.raises(NotImplementedError):
        UNetModel(32, 4, 320, 4, 2, [4, 2, 1], num_heads=8, use_spatial_transformer=False)


def test_weight_recipe_is_deterministic():
    from adaprompt_b200.weights import synth_state_dict
    spec = {"a.weight": (8, 4, 3, 3), "a.bias": (8,), "n.weight": (8,), "n.bias": (8,)}
    s1, s2 = synth_state_dict(spec, 7), synth_state_dict(spec, 7)
    assert all(torch.equal(s1[k], s2[k]) for k in spec)
    assert not torch.equal(s1["a.weight"], synth_state_dict(spec, 8)["a.weight"])
    assert s1["a.weight"].abs().max() <= 1 / 6.0 + 1e-6 and abs(s1["n.weight"].mean() - 1) < 0.1


def test_gemm_and_conv_schedule_plans():
    """af_gemm_plan / af_conv3x3_plan: the tile width, CTA-pair and split-K decisions of the GEMM / conv kernel for the
    UNet's shapes at the benchmarked batch (no device needed: 148 SMs are assumed).  These are the measured rules of
    profiles/r02_splitk.md - a change of a rule has to show up here."""
    import ctypes
    from adaprompt_b200 import _lib
    lib = _lib.load()
    WS = 16384 + 48 * (1 << 20)

    def ep(res=False, geglu=False, bf16=False, ws=True, split_k=0, pair_mode=0):
        e = _lib.AfEpilogue()
        e.out_dtype = 1 if bf16 else 0
        e.geglu = 1 if geglu else 0
        e.split_k, e.pair_mode = split_k, pair_mode
        if res:
            e.residual = 1            # only tested for NULL by the planner
        if ws:
            e.splitk_ws, e.splitk_ws_bytes = 1, WS
        return e

    def conv(C0, C1, B, H, Cout, stride=1, **kw):
        out = (ctypes.c_int * 6)()
        e = ep(**kw)
        assert lib.af_conv3x3_plan(C0, C1, B, H, H, Cout, stride, ctypes.byref(e), 0, out) == 0
        return dict(zip(("bn", "pair", "split", "units", "dp", "wide"), out))

    def gemm(M, N, K, **kw):
        out = (ctypes.c_int * 6)()
        e = ep(**kw)
        assert lib.af_gemm_plan(M, N, K, ctypes.byref(e), 0, out) == 0
        return dict(zip(("bn", "pair", "split", "units", "dp", "wide"), out))

    # 8x8 convolutions: 64 tiles on 148 SMs -> two K ranges each fill one wave; no pairs
    p = conv(1280, 0, 16, 8, 1280, res=True)
    assert (p["bn"], p["pair"], p["split"], p["units"], p["dp"]) == (160, 0, 2, 128, 0)
    assert conv(1280, 0, 16, 8, 1280, res=True, ws=False)["split"] == 1          # no workspace: whole tiles
    assert conv(1280, 0, 16, 8, 1280, res=True, split_k=1)["split"] == 1         # per-call override
    # 16x16 convolutions to 1280 channels: 256-wide tiles, one full wave + 12 split remainder tiles
    p = conv(1280, 0, 16, 16, 1280, res=True)
    assert (p["bn"], p["pair"], p["dp"]) == (256, 0, 148) and p["split"] > 1 and p["units"] == 148 + 12 * p["split"]
    # 64x64 / 32x32 stride-1 convolutions with 160-wide tiles: CTA pairs, whole tiles
    for args in ((320, 0, 16, 64, 320), (640, 320, 16, 64, 320), (640, 0, 16, 32, 640)):
        p = conv(*args, res=True)
        assert (p["bn"], p["pair"], p["split"]) == (160, 1, 1), (args, p)
    assert conv(320, 0, 16, 64, 320, stride=2)["pair"] == 1                     # the 64 -> 32 downsample has 128 row tiles too
    assert conv(640, 0, 16, 32, 640, stride=2)["pair"] == 0                     # 32 row tiles: single-CTA tiles
    assert conv(128, 0, 8, 512, 128)["pair"] == 1                               # VAE decoder: >= 512 row tiles
    # linear GEMMs: 160 for the short-K residual projections, 256 where K dominates, pairs from 16 row tiles
    assert gemm(65536, 320, 320, res=True) == dict(bn=160, pair=1, split=1, units=1024, dp=1024, wide=0)
    p = gemm(4096, 1280, 5120, res=True)
    assert (p["bn"], p["pair"], p["split"]) == (256, 1, 1)
    p = gemm(1024, 1280, 5120, res=True)                                        # 8 row tiles: no pairs, split-K instead
    assert (p["bn"], p["pair"]) == (256, 0) and p["split"] == 2
    assert gemm(1024, 1280, 1280, res=True)["split"] == 1                       # short K: splitting only adds overhead
    p = gemm(65536, 768, 320, bf16=True)                                        # fused QK projection: wide bf16 epilogue
    assert (p["bn"], p["wide"]) == (256, 1)
    assert gemm(65536, 320, 320, bf16=True)["wide"] == 0                        # 160-wide tiles keep 32-column items
    assert gemm(4096, 10240, 1280, geglu=True, bf16=True)["bn"] == 256


@pytest.mark.parametrize("call,message", [
    (("gemm", 4096, 324, 320, {}), b"af_gemm_bf16: N=324 must be a multiple of 8"),
    (("gemm", 4096, 10240, 1280, dict(geglu=1, residual=16)), b"geglu epilogue: residual / rowbias unsupported"),
    (("gemm", 4096, 10112, 1280, dict(geglu=1)), b"geglu: packed N=10112 must be a multiple of 256"),
    (("gemm", 4096, 10240, 1280, dict(geglu=1, act=1)), b"epilogue: act 1 unsupported"),
    (("conv", 100, 0, 16, 32, 32, 320, 1), b"af_conv3x3_bf16: C0=100 C1=0 must each be a multiple of 64"),
    (("conv", 320, 0, 16, 32, 32, 320, 3), b"af_conv3x3_bf16: stride 3"),
    (("conv", 320, 0, 16, 33, 32, 320, 2), b"af_conv3x3_bf16: stride 2 needs a single source and even H=33 W=32"),
], ids=["gemm-N%8", "geglu-residual", "geglu-N%256", "geglu-act", "conv-C0=100", "conv-stride3", "conv-s2-oddH"])
def test_schedule_plans_refuse_what_the_launch_refuses(call, message):
    """af_gemm_plan / af_conv3x3_plan run the argument checks of af_gemm_bf16 / af_conv3x3_bf16: sizes or epilogue
    options the launch refuses get no schedule, but the launch's negative code and message."""
    import ctypes
    from adaprompt_b200 import _lib
    lib = _lib.load()
    out = (ctypes.c_int * 6)()
    e = _lib.AfEpilogue()
    e.out_dtype = 1                     # bf16, as GEGLU needs
    if call[0] == "gemm":
        M, N, K, fields = call[1:]
        for k, v in fields.items():
            setattr(e, k, v)            # residual: only tested for NULL by the planner
        rc = lib.af_gemm_plan(M, N, K, ctypes.byref(e), 0, out)
    else:
        rc = lib.af_conv3x3_plan(*call[1:], ctypes.byref(e), 0, out)
    assert rc < 0
    assert lib.af_last_error() == message
