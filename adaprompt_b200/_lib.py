"""ctypes binding of libadaface_b200.so (include/adaface_b200.h).

The product path has no CPU fallback: if the library is missing, or there is no sm_100 device,
every op raises.  The library itself loads fine on a CPU-only box (static cudart, driver entry
points resolved lazily) so that symbol-export checks can run without a GPU.
"""
from __future__ import annotations

import ctypes
import os
import types
from ctypes import POINTER, Structure, c_char_p, c_float, c_int, c_longlong, c_size_t, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libadaface_b200.so")

AF_DTYPE_F32 = 0
AF_DTYPE_BF16 = 1


class AfEpilogue(Structure):
    _fields_ = [
        ("bias", c_void_p),
        ("rowbias", c_void_p),
        ("rows_per_group", c_int),
        ("ld_rowbias", c_longlong),
        ("residual", c_void_p),
        ("ldr", c_longlong),
        ("out", c_void_p),
        ("ldo", c_longlong),
        ("out_dtype", c_int),
        ("geglu", c_int),
        ("act", c_int),
        ("gn_stats", c_void_p),
        ("pair_mode", c_int),
        ("trace", c_void_p),
        ("splitk_ws", c_void_p),
        ("splitk_ws_bytes", c_longlong),
        ("split_k", c_int),
    ]


class AfBgemm(Structure):
    _fields_ = [
        ("A", c_void_p), ("lda", c_longlong), ("sA0", c_longlong), ("sA1", c_longlong),
        ("B", c_void_p), ("ldb", c_longlong), ("sB0", c_longlong), ("sB1", c_longlong),
        ("C", c_void_p), ("ldc", c_longlong), ("sC0", c_longlong), ("sC1", c_longlong), ("c_dtype", c_int),
        ("vec", c_void_p), ("sV0", c_longlong), ("sV1", c_longlong),
        ("P", c_void_p), ("ldp", c_longlong), ("sP0", c_longlong), ("sP1", c_longlong),
        ("M", c_int), ("N", c_int), ("K", c_int), ("nb0", c_int), ("nb1", c_int), ("mode", c_int),
        ("valid_rows", c_int), ("valid_cols", c_int), ("alpha", c_float),
    ]


# symbol -> (restype, argtypes); mirrors include/adaface_b200.h one to one
SIGNATURES = {
    "af_version": (c_int, []),
    "af_last_error": (c_char_p, []),
    "af_device_info": (c_int, [POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "af_gemm_bf16": (c_int, [c_void_p, c_longlong, c_int, c_void_p, c_longlong, c_int, c_void_p, c_int, c_int,
                             POINTER(AfEpilogue), c_int, c_void_p]),
    "af_conv3x3_bf16": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                POINTER(AfEpilogue), c_int, c_void_p]),
    "af_gemm_plan": (c_int, [c_int, c_int, c_int, POINTER(AfEpilogue), c_int, POINTER(c_int)]),
    "af_conv3x3_plan": (c_int, [c_int, c_int, c_int, c_int, c_int, c_int, c_int, POINTER(AfEpilogue), c_int,
                                POINTER(c_int)]),
    "af_attention_bf16": (c_int, [c_void_p, c_longlong, c_void_p, c_longlong, c_void_p, c_longlong, c_int, c_void_p,
                                  c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "af_conv3x3_gn_slots": (c_int, [c_int, c_int]),
    "af_conv3x3_down01_bf16": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, POINTER(AfEpilogue),
                                       c_int, c_void_p]),
    "af_xattn_explicit": (c_int, [c_void_p, c_longlong, c_void_p, c_longlong, c_void_p, c_longlong, c_int, c_void_p, c_void_p,
                                  c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "af_conv_attn_scores": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "af_attention_bwd_bf16": (c_int, [c_void_p, c_longlong, c_void_p, c_longlong, c_void_p, c_longlong, c_void_p, c_longlong,
                                      c_void_p, c_longlong, c_void_p, c_longlong, c_void_p, c_longlong, c_void_p, c_void_p,
                                      c_void_p, c_longlong, c_void_p, c_longlong, c_void_p, c_longlong, c_int, c_int, c_int,
                                      c_int, c_void_p]),
    "af_attention_bf16_trace": (c_int, [c_void_p, c_longlong, c_void_p, c_longlong, c_void_p, c_longlong, c_int, c_void_p,
                                        c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "af_groupnorm_workspace_bytes": (c_size_t, [c_int, c_int]),
    "af_groupnorm_stats_slots": (c_int, [c_int, c_int]),
    "af_groupnorm_stats": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_void_p]),
    "af_groupnorm_finalize": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p,
                                      c_void_p]),
    "af_groupnorm_apply": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int,
                                   c_void_p, c_void_p, c_void_p]),
    "af_groupnorm_silu": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_float, c_int,
                                  c_void_p, c_void_p, c_void_p, c_void_p]),
    "af_layernorm": (c_int, [c_void_p, c_longlong, c_int, c_void_p, c_void_p, c_float, c_void_p, c_void_p]),
    "af_layernorm_f32": (c_int, [c_void_p, c_longlong, c_int, c_void_p, c_void_p, c_float, c_void_p, c_void_p]),
    "af_conv_in": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "af_conv_out": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "af_nhwc_to_nchw": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "af_timestep_embedding": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "af_linear_small": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "af_cast_bf16": (c_int, [c_void_p, c_void_p, c_longlong, c_void_p]),
    "af_upsample2x_cast": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "af_cfg_ddim_update": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_longlong, c_void_p]),
    "af_advance_step": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "af_attention_small": (c_int, [c_void_p, c_longlong, c_int, c_int, c_void_p, c_longlong, c_int, c_int, c_int, c_int,
                                   c_float, c_int, c_void_p]),
    "af_gather_rows": (c_int, [c_void_p, c_void_p, c_void_p, c_longlong, c_int, c_int, c_void_p]),
    "af_add_pos": (c_int, [c_void_p, c_void_p, c_longlong, c_int, c_int, c_void_p]),
    "af_find_first_token": (c_int, [c_void_p, c_int, c_int, c_longlong, c_void_p, c_void_p]),
    "af_splice_rows": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "af_weighted_sum": (c_int, [c_void_p, c_void_p, c_void_p, c_float, c_float, c_float, c_void_p, c_longlong,
                                c_void_p]),
    # ---- training step (backward kernels)
    "af_attention_bf16_lse": (c_int, [c_void_p, c_longlong, c_void_p, c_longlong, c_void_p, c_longlong, c_int,
                                      c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "af_bgemm_bf16": (c_int, [POINTER(AfBgemm), c_void_p]),
    "af_groupnorm_bwd_workspace_floats": (c_size_t, [c_int, c_int, c_int]),
    "af_groupnorm_bwd": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p,
                                 c_void_p, c_void_p, c_void_p, c_void_p]),
    "af_layernorm_bwd": (c_int, [c_void_p, c_longlong, c_int, c_void_p, c_float, c_void_p, c_int, c_void_p, c_void_p,
                                 c_void_p, c_void_p, c_void_p]),
    "af_geglu_fwd": (c_int, [c_void_p, c_longlong, c_int, c_void_p, c_void_p]),
    "af_geglu_bwd": (c_int, [c_void_p, c_void_p, c_longlong, c_int, c_void_p, c_void_p]),
    "af_quick_gelu": (c_int, [c_void_p, c_void_p, c_longlong, c_void_p, c_void_p]),
    "af_rowdot_heads": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "af_attention_small_bwd": (c_int, [c_void_p, c_longlong, c_int, c_int, c_void_p, c_longlong, c_void_p, c_int,
                                       c_int, c_int, c_int, c_float, c_int, c_void_p]),
    "af_conv_out_dgrad": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "af_sumpool2x2": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "af_zero_insert2x": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "af_transpose_to_bf16": (c_int, [c_void_p, c_int, c_int, c_int, c_longlong, c_void_p, c_void_p]),
    "af_channel_mix4": (c_int, [c_void_p, c_void_p, c_void_p, c_float, c_int, c_int, c_int, c_longlong, c_void_p, c_void_p]),
    "af_softmax_rows": (c_int, [c_void_p, c_longlong, c_longlong, c_int, c_float, c_void_p, c_longlong, c_void_p]),
    "af_vae_posterior": (c_int, [c_void_p, c_int, c_longlong, c_int, c_void_p, c_float, c_void_p, c_void_p, c_void_p,
                                 c_void_p]),
    "af_prodigy_moments": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_longlong, c_float,
                                   c_float, c_float, c_float, c_float, c_float, c_void_p, c_void_p]),
    "af_prodigy_apply": (c_int, [c_void_p, c_void_p, c_void_p, c_longlong, c_float, c_float, c_float, c_void_p]),
}

_lib = None


class AdaFaceB200Error(RuntimeError):
    pass


ABI_VERSION = 202      # include/adaface_b200.h AF_VERSION


def load():
    """Loads the shared library (building is the job of __graft_entry__.build / adaprompt_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise AdaFaceB200Error(
            f"{LIB_PATH} not found: build it with `python -m adaprompt_b200.build` (needs nvcc, sm_100a). "
            "There is no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    lib.af_version.restype = c_int
    if lib.af_version() != ABI_VERSION:        # a stale build: struct layouts (af_epilogue) would not match this binding
        raise AdaFaceB200Error(f"{LIB_PATH} has ABI version {lib.af_version()}, this binding needs {ABI_VERSION}: rebuild "
                               "with `python -m adaprompt_b200.build`")
    ns = types.SimpleNamespace(_cdll=lib)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
        setattr(ns, name, _traced(name, fn) if name in KERNELS_PER_CALL else fn)
    _lib = ns
    return ns


# ---------------------------------------------------------------------------------------------------
# launch accounting / per-launch timing (bench.py: gpu_launches, roofline; no effect on results)
# ---------------------------------------------------------------------------------------------------
KERNELS_PER_CALL = {
    "af_gemm_bf16": 1, "af_conv3x3_bf16": 1, "af_attention_bf16": 1, "af_groupnorm_silu": 3, "af_layernorm": 1,
    "af_groupnorm_stats": 1, "af_groupnorm_finalize": 1, "af_groupnorm_apply": 1, "af_nhwc_to_nchw": 1,
    "af_attention_small": 1, "af_gather_rows": 1, "af_add_pos": 1, "af_find_first_token": 1, "af_splice_rows": 1,
    "af_weighted_sum": 1, "af_layernorm_f32": 1,
    "af_conv_in": 1, "af_conv_out": 1, "af_timestep_embedding": 1, "af_linear_small": 1, "af_cast_bf16": 1,
    "af_upsample2x_cast": 1, "af_cfg_ddim_update": 1, "af_advance_step": 1,
    "af_attention_bf16_lse": 1, "af_attention_bwd_bf16": 2, "af_xattn_explicit": 1, "af_conv_attn_scores": 1, "af_bgemm_bf16": 1, "af_groupnorm_bwd": 3, "af_layernorm_bwd": 1, "af_geglu_fwd": 1,
    "af_geglu_bwd": 1, "af_quick_gelu": 1, "af_rowdot_heads": 1, "af_attention_small_bwd": 1, "af_conv_out_dgrad": 1,
    "af_sumpool2x2": 1, "af_zero_insert2x": 1, "af_transpose_to_bf16": 1, "af_prodigy_moments": 1, "af_prodigy_apply": 1,
    "af_softmax_rows": 1, "af_channel_mix4": 1, "af_conv3x3_down01_bf16": 1, "af_vae_posterior": 1,
}


def _cost(name, a):
    """(algorithmic flops, algorithmic bytes) of one call, from its C arguments."""
    if name == "af_gemm_bf16":
        K, M, N = a[2] + a[5], a[7], a[8]
        ep = a[9]._obj
        No = N // 2 if ep.geglu else N
        by = 2.0 * (M * K + N * K) + (4.0 if ep.out_dtype == 0 else 2.0) * M * No + (4.0 * M * No if ep.residual else 0.0)
        return 2.0 * M * N * K, by
    if name == "af_conv3x3_bf16":
        C, B, H, W, Co, s = a[1] + a[3], a[5], a[6], a[7], a[8], a[9]
        px = B * (H // s) * (W // s)
        ep = a[10]._obj
        by = 2.0 * (B * H * W * C + 9 * C * Co) + (4.0 if ep.out_dtype == 0 else 2.0) * px * Co \
            + (4.0 * px * Co if ep.residual else 0.0)
        return 2.0 * px * Co * 9 * C, by
    if name == "af_attention_bf16":
        B, h, Nq, Nk, d = a[9], a[10], a[11], a[12], a[13]
        return 4.0 * B * h * Nq * Nk * d, 2.0 * B * h * d * (2 * Nq + 2 * Nk)
    if name == "af_groupnorm_silu":
        n = a[4] * a[5] * (a[1] + a[3])
        return 8.0 * n, 6.0 * n + (2.0 * n if a[11] else 0.0)
    if name == "af_groupnorm_apply":
        n = a[4] * a[5] * (a[1] + a[3])
        return 8.0 * n, 6.0 * n + (2.0 * n if a[11] else 0.0)
    if name == "af_groupnorm_stats":
        return 0.0, 0.0  # overhead pass: its bytes are not algorithmic (the 6 B/element are charged to apply)
    if name == "af_layernorm":
        n = a[1] * a[2]
        return 8.0 * n, 6.0 * n
    return 0.0, 0.0


def _sig(name, a):
    """Shape signature of one call (per-shape breakdown in bench.py --breakdown)."""
    if name == "af_gemm_bf16":
        ep = a[9]._obj
        return f"M{a[7]} N{a[8]} K{a[2] + a[5]}{' geglu' if ep.geglu else ''}{' res' if ep.residual else ''}" \
               f"{' f32' if ep.out_dtype == 0 else ''}"
    if name == "af_bgemm_bf16":
        g = a[0]._obj
        return f"M{g.M} N{g.N} K{g.K} nb{g.nb0}x{g.nb1} mode{g.mode}"
    if name == "af_conv3x3_bf16":
        return f"B{a[5]} {a[6]}x{a[7]} C{a[1] + a[3]}->{a[8]} s{a[9]}"
    if name == "af_attention_bf16":
        return f"B{a[9]} Nq{a[11]} Nk{a[12]} d{a[13]}"
    if name in ("af_groupnorm_silu", "af_groupnorm_apply"):
        return f"B{a[4]} HW{a[5]} C{a[1] + a[3]}"
    if name == "af_layernorm":
        return f"rows{a[1]} C{a[2]}"
    return ""


class _Trace:
    count = 0          # kernels launched through the C ABI since import
    records = None     # list of (name, start_event, end_event, flops, bytes) while profiling


TRACE = _Trace()


def _traced(name, fn):
    nk = KERNELS_PER_CALL[name]

    def call(*args):
        TRACE.count += nk
        if TRACE.records is None:
            return fn(*args)
        import torch
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        rc = fn(*args)
        e1.record()
        fl, by = _cost(name, args)
        TRACE.records.append((name, e0, e1, fl, by, _sig(name, args)))
        return rc

    call.__name__ = name
    return call


class profile:
    """with _lib.profile() as recs: ...  -> recs.summary() after a synchronize: per-entry-point launch count,
    total device ms (CUDA events on the launching stream), algorithmic flops / bytes."""

    def __enter__(self):
        TRACE.records = []
        self.records = TRACE.records
        return self

    def __exit__(self, *exc):
        TRACE.records = None
        return False

    def summary(self):
        import torch
        torch.cuda.synchronize()
        out = {}
        self.by_shape = {}
        for name, e0, e1, fl, by, sig in self.records:
            ms = e0.elapsed_time(e1)
            for table, key in ((out, name), (self.by_shape, f"{name[3:]} {sig}")):
                d = table.setdefault(key, {"launches": 0, "ms": 0.0, "flops": 0.0, "bytes": 0.0})
                d["launches"] += 1
                d["ms"] += ms
                d["flops"] += fl
                d["bytes"] += by
        return out


SYNC_DEBUG = os.environ.get("AF_SYNC_DEBUG", "0") == "1"


def check(rc: int, what: str) -> None:
    if rc == 0:
        if SYNC_DEBUG:  # debugging aid: surface asynchronous kernel faults at the launch that caused them
            import torch
            try:
                torch.cuda.synchronize()
            except Exception as e:  # noqa: BLE001
                raise AdaFaceB200Error(f"{what}: kernel fault detected right after launch: {e}") from e
        return
    msg = load().af_last_error().decode(errors="replace")
    if rc < 0:
        raise ValueError(f"{what}: {msg} (rc={rc})")
    raise AdaFaceB200Error(f"{what}: {msg} (cudaError {rc})")
