"""GroupNorm(32) [+SiLU] and LayerNorm kernels, forward and backward, against the float64 references of
tests/norm_reference.py, with per-(sample, group) and per-row limits; plus the elementwise kernels of the training step.

Each GroupNorm producer of statistics (the stand-alone pass, the GEMM epilogue, the conv epilogue) is checked per
(sample, group) mean and rstd; the apply and backward kernels are checked per group, LayerNorm per row.  Inputs come
from the regimes of norm_reference.gn_input / ln_input: iid, structured (every slot, channel and sample contributes a
distinguishable amount), offset (a large group mean next to its std) and degenerate.  In the structured regime each
test also shows that its limit sits at least 5x below the error of a plausible bookkeeping defect (a statistic that
skips the last slot or chunk, a channel reading the next group's statistics, a sample reading the next sample's).

Limits are about twice the worst values observed on a B200 (1000 W power limit); the observed values are beside them.
Sources of error: bf16 rounding of the outputs (relative 2^-9 at most, ~2^-9/sqrt(3) RMS), fp32 accumulation, and the
one-pass variance E[x^2] - E[x]^2 of the GroupNorm statistics, whose relative rstd error grows with (mean/std)^2."""
import contextlib

import pytest
import torch

import norm_reference as nr

pytestmark = pytest.mark.gpu

DEV = "cuda"

# ---- limits: about twice the worst value observed on a B200 (1000 W power limit), observed worst in brackets
STATS_MEAN = 1e-6          # mean error in units of sqrt(var + eps), iid / structured / degenerate / conv  [5.1e-7]
STATS_RSTD = 4e-6          # relative rstd error, same regimes                                          [2.1e-6]
# one-pass variance: relative rstd error at mean/std = 30 and 100 [1.8e-4, 1.4e-3]; at 300 it reaches 1.5e-2 (recorded,
# not asserted).  Mean error in std units [4.9e-6, 1.3e-5].
OFFSET_RSTD = {30: 3.5e-4, 100: 2.7e-3}
OFFSET_MEAN = {30: 1e-5, 100: 3e-5}
GN_OUT_GROUP = 4.5e-3      # bf16 GroupNorm output, worst (sample, group), also at mean/std 30 and 100   [2.2e-3; 1.7e-3, 2.3e-3]
GN_OUT_REL = 3.5e-3        # bf16 GroupNorm output, global rel-L2                                       [1.7e-3]
GN_BWD_GROUP = 1.2e-6      # dx of the backward kernels fed the reference statistics, worst group       [6.0e-7]
GN_BWD_SUM = 1.2e-6        # |sum_group dx| / sum_group |dx| without dres                               [5.6e-7]
GN_FN_GROUP = 1.1e-6       # GroupNormFn dx (kernel statistics) against the exact-statistics reference  [5.4e-7]
# bf16 LayerNorm output, worst row: bf16 rounding alone reaches 2^-8 relative per value, and a row of 4 values gets
# close to it [3.5e-3 at C = 4, 1.9e-3 at C = 2048, both what rounding the float64 result gives].  A bf16 row cannot
# resolve one dropped float4 of 2048 channels 5x over, so the sensitivity of the kernel template's statistics is
# asserted through its fp32-output instantiations.
LN_BF16_ROW = 4e-3
LN_F32_ROW = 1e-6          # fp32 LayerNorm output, worst row (iid / structured), at C = 4          [4.6e-7]
# fp32 LayerNorm output at mean/std 30 and 1000: the sum of the row loses ~1000 ulp of its std, and a row of 4 values
# can have a sample std well below that of its distribution                                                  [6.9e-4]
LN_F32_ROW_OFFSET = 1.4e-3
LN_BWD_ROW = 8e-7          # LayerNorm dx, worst row                                                    [3.8e-7]
LN_BWD_SUM = 4e-7          # |sum_row dx| / sum_row |dx| without dres                                   [1.6e-7]
LN_PARAM_REL = 3e-6        # dgamma / dbeta rel-L2                                                      [1.5e-6]
SENS = 5.0                 # each limit sits this far below the error of a modelled defect

OBSERVED = {}


def _seen(key, value):
    OBSERVED[key] = max(OBSERVED.get(key, 0.0), value)
    return value


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    yield
    print("\nnorm tests, worst observed: " + "  ".join(f"{k} {v:.3e}" for k, v in sorted(OBSERVED.items())))


def _stream():
    return torch.cuda.current_stream().cuda_stream


@contextlib.contextmanager
def _kernels():
    """Collects the names (spaces removed) of the CUDA kernels that ran inside the block."""
    names = []
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        yield names
        torch.cuda.synchronize()
    names.extend(e.key.replace(" ", "") for e in prof.key_averages())


def _sens_check(label, limit, sens):
    for k, s in sens.items():
        assert SENS * limit < s, f"{label}: limit {limit} would not catch the '{k}' defect ({s:.3e})"


def _default_slots(B, HW):
    from adaprompt_b200 import _lib
    return _lib.load().af_groupnorm_stats_slots(B, HW)


def _bwd_chunks(B, HW):
    """The chunk count af_groupnorm_bwd picks (train.cu gn_bwd_chunks), for the defect model."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    return max(1, min((4 * sms + B - 1) // B, HW // 16, 256))


def _check_stats(label, x, mr, eps, slots, regime, mean_lim=STATS_MEAN, rstd_lim=STATS_RSTD):
    mean, rstd = nr.gn_stats_ref(x, eps)
    e = nr.stats_errors(mr, mean, rstd)
    _seen(f"stats_mean[{regime}]", e["mean"])
    _seen(f"stats_rstd[{regime}]", e["rstd"])
    if regime == "structured":
        _sens_check(label, max(mean_lim, rstd_lim), nr.gn_stats_sensitivity(x, eps, slots))
    assert e["mean"] < mean_lim and e["rstd"] < rstd_lim, (label, e)
    return e


# ------------------------------------------------------------------------------------------------ GroupNorm statistics
STATS_CASES = [  # C, HW, B, regime: every lane width (C 128..960: 8/4/2/3/1 pixel lanes; wider: channel loop), HW with
    # a single slot (1, 15), uneven slots (100, 1000: trailing slots empty), full 64 slots (1536, 4096, 9216), B to 16
    (128, 1000, 2, "structured"), (128, 4096, 16, "structured"), (256, 100, 16, "structured"), (256, 1, 1, "iid"),
    (512, 1536, 1, "structured"), (512, 15, 2, "iid"), (320, 4096, 2, "structured"), (320, 9216, 1, "structured"),
    (640, 1000, 1, "structured"), (640, 15, 16, "structured"), (960, 15, 2, "structured"), (960, 1000, 2, "iid"),
    (1280, 1, 16, "structured"), (1280, 1536, 2, "structured"), (1920, 100, 2, "structured"),
    (2560, 1000, 1, "structured"), (2560, 100, 16, "structured"), (5120, 15, 2, "structured"),
    (5120, 100, 1, "structured"), (5120, 1, 16, "iid"), (320, 1000, 2, "degenerate"), (1280, 100, 1, "degenerate"),
]


@pytest.mark.parametrize("C,HW,B,regime", STATS_CASES)
def test_groupnorm_stats_pass(C, HW, B, regime):
    from adaprompt_b200 import ops
    x = nr.gn_input(regime, B, HW, C, seed=C + HW + B, device=DEV)
    for eps in (1e-5, 1e-6):
        st = ops.groupnorm_stats(x)
        _check_stats(f"C={C} HW={HW} B={B} {regime}", x, ops.groupnorm_mean_rstd(x, st, eps), eps, st.slots, regime)


@pytest.mark.parametrize("C,HW,B,slots", [
    (320, 1000, 2, 1), (320, 100, 2, 100), (320, 1000, 2, 62), (128, 1000, 1, 62), (2560, 1000, 1, 59),
    (640, 15, 2, 15), (5120, 100, 2, 7), (960, 4096, 1, 64), (256, 9216, 1, 64), (1280, 1000, 16, 62),
])
def test_groupnorm_stats_explicit_slots(C, HW, B, slots):
    """af_groupnorm_stats with a caller-chosen slot count: one slot, one pixel per slot, and ceil(HW / slots) pixels
    per slot with a short last slot or empty trailing slots (HW = 1000, 62 slots: 17 pixels each, the last three
    empty)."""
    from adaprompt_b200 import _lib, ops
    lib = _lib.load()
    x = nr.gn_input("structured", B, HW, C, seed=3, device=DEV)
    buf = torch.full((B * slots * C * 2,), float("nan"), device=DEV)
    assert lib.af_groupnorm_stats(x.data_ptr(), C, B, HW, buf.data_ptr(), slots, _stream()) == 0
    part = buf.reshape(B, slots, C, 2).double()
    assert torch.isfinite(part).all()
    for s, (p0, p1) in enumerate(nr.slot_bounds(HW, slots)):     # every slot holds exactly its own pixels
        xs = x[:, p0:p1].double()
        assert torch.allclose(part[:, s, :, 0], xs.sum(1), rtol=1e-5, atol=1e-4 * (p1 - p0 + 1)), s
        assert torch.allclose(part[:, s, :, 1], (xs * xs).sum(1), rtol=1e-5, atol=1e-4 * (p1 - p0 + 1)), s
    mr = ops.groupnorm_mean_rstd(x, ops.GNStats(buf, slots, C), 1e-5)
    _check_stats(f"C={C} HW={HW} B={B} slots={slots}", x, mr, 1e-5, slots, "structured")


@pytest.mark.parametrize("k", [30, 100, 300])
def test_groupnorm_offset_regime(k):
    """Groups whose mean is k times their std, through the stand-alone statistics pass and through the GEMM epilogue.
    The one-pass variance loses accuracy as (mean/std)^2: the rstd error has its own limit at 30 and at 100 and is only
    recorded at 300; up to 100 the bf16 output still meets the iid limit."""
    from adaprompt_b200 import ops
    B, HW, C, eps = 2, 1024, 640, 1e-5
    x = nr.gn_input(f"offset{k}", B, HW, C, seed=k, device=DEV)
    gamma, beta = nr.affine(C, 1, DEV)
    # the same tensor as a GEMM output: identity weights, x as the residual (the epilogue writes exactly x)
    a = torch.zeros(B * HW, 64, dtype=torch.bfloat16, device=DEV)
    w = torch.zeros(C, 64, dtype=torch.bfloat16, device=DEV)
    out = torch.empty(B * HW, C, device=DEV)
    st_g = ops.gn_stats_for_gemm(B, HW, C, DEV)
    ops.gemm(a, w, out, residual=x.reshape(B * HW, C), gn_stats=st_g.buf)
    assert torch.equal(out.reshape(B, HW, C), x)
    y_ref, mean, rstd = nr.gn_ref(x, None, gamma, beta, eps, True)
    for name, st in (("stats pass", ops.groupnorm_stats(x)), ("gemm epilogue", st_g)):
        e = nr.stats_errors(ops.groupnorm_mean_rstd(x, st, eps), mean, rstd)
        y = torch.empty(B, HW, C, dtype=torch.bfloat16, device=DEV)
        ops.groupnorm_apply(x, st, gamma, beta, eps, True, y)
        wg = nr.worst_group(y, y_ref)
        _seen(f"offset{k}_rstd", e["rstd"])
        _seen(f"offset{k}_mean", e["mean"])
        _seen(f"offset{k}_out_group", wg)
        print(f"\nmean/std {k} {name}: rstd {e['rstd']:.3e} mean {e['mean']:.3e} output group {wg:.3e}")
        if k in OFFSET_RSTD:
            assert e["rstd"] < OFFSET_RSTD[k] and e["mean"] < OFFSET_MEAN[k], (name, e)
            assert wg < GN_OUT_GROUP, (name, wg)


@pytest.mark.parametrize("B,HW,N,regime", [(2, 4096, 320, "structured"), (3, 256, 1280, "structured"),
                                           (16, 64, 640, "structured"), (1, 1024, 2560, "iid"), (2, 96, 5120, "structured")])
def test_groupnorm_stats_from_gemm_epilogue(B, HW, N, regime):
    """The GEMM epilogue's per-32-row statistics, folded by gn_finalize_kernel, against float64 statistics of the tensor
    the GEMM wrote; the structure reaches the output through the residual."""
    from adaprompt_b200 import ops
    M, K = B * HW, 128
    g = torch.Generator().manual_seed(N)
    a = (torch.randn(M, K, generator=g) * 0.5).to(torch.bfloat16).to(DEV)
    w = (torch.randn(N, K, generator=g) * K ** -0.5).to(torch.bfloat16).to(DEV)
    bias = (torch.randn(N, generator=g) * 0.3).to(DEV)
    res = nr.gn_input(regime, B, HW, N, seed=N + 1, device=DEV).reshape(M, N)
    out = torch.empty(M, N, device=DEV)
    st = ops.gn_stats_for_gemm(B, HW, N, DEV)
    ops.gemm(a, w, out, bias=bias, residual=res, gn_stats=st.buf)
    x = out.reshape(B, HW, N)
    _check_stats(f"gemm B={B} HW={HW} N={N}", x, ops.groupnorm_mean_rstd(x, st, 1e-5), 1e-5, st.slots, regime)


@pytest.mark.parametrize("mode,B,H,W,Cin,Cout", [("stride1", 2, 24, 24, 320, 320), ("stride1", 2, 64, 64, 320, 640),
                                                 ("stride2", 2, 32, 32, 640, 640), ("down01", 2, 48, 48, 128, 128),
                                                 ("down01", 1, 64, 64, 256, 256)])
def test_groupnorm_stats_from_conv_epilogue(mode, B, H, W, Cin, Cout):
    """The conv epilogue's statistics (one slot per 32 pixels of a tile box; a 24x24 or 24x24-output image leaves boxes
    that overhang it) against float64 statistics of the conv output.  The input carries a per-pixel ramp and a
    per-sample scale, the bias distinct per-channel offsets."""
    from adaprompt_b200 import ops
    from adaprompt_b200.packing import pack_conv3x3
    g = torch.Generator().manual_seed(Cin + H)
    ramp = torch.linspace(0.2, 2.0, H * W).reshape(1, H, W, 1) ** 2
    scale = (1 + 0.5 * torch.arange(B, dtype=torch.float32)).reshape(B, 1, 1, 1)
    x = (torch.randn(B, H, W, Cin, generator=g) * ramp * scale).to(torch.bfloat16).to(DEV)
    w = (torch.randn(Cout, Cin, 3, 3, generator=g) * (9 * Cin) ** -0.5).to(DEV)
    bias = (torch.randn(Cout, generator=g) * 2).to(DEV)
    Ho, Wo = H // 2 if mode != "stride1" else H, W // 2 if mode != "stride1" else W
    out = torch.empty(B, Ho, Wo, Cout, device=DEV)
    st = ops.gn_stats_for_conv(B, Ho, Wo, Cout, DEV)
    assert st is not None
    if mode == "down01":
        ops.conv3x3_down01(x, pack_conv3x3(w), out, bias=bias, gn_stats=st.buf)
    else:
        res = nr.gn_input("structured", B, Ho * Wo, Cout, seed=5, device=DEV).reshape(B, Ho, Wo, Cout)
        ops.conv3x3(x, pack_conv3x3(w), out, stride=1 if mode == "stride1" else 2, bias=bias, residual=res,
                    gn_stats=st.buf)
    xo = out.reshape(B, Ho * Wo, Cout)
    mean, rstd = nr.gn_stats_ref(xo, 1e-6)
    e = nr.stats_errors(ops.groupnorm_mean_rstd(xo, st, 1e-6), mean, rstd)
    _seen("stats_mean[conv]", e["mean"])
    _seen("stats_rstd[conv]", e["rstd"])
    assert e["mean"] < STATS_MEAN and e["rstd"] < STATS_RSTD, e


# ------------------------------------------------------------------------------------------------ GroupNorm apply
APPLY_CASES = [  # B, HW, C0, C1, eps, silu, regime.  640 | 320 and 1280 | 640: group 21 straddles the two sources;
    # HW * C / 4 not a multiple of 1024 in most cases (per-block tail of gn_apply_kernel)
    (2, 100, 640, 320, 1e-5, True, "structured"), (1, 1000, 1280, 640, 1e-6, False, "structured"),
    (2, 15, 960, 0, 1e-5, True, "iid"), (16, 64, 1280, 1280, 1e-5, True, "structured"),
    (2, 4096, 320, 0, 1e-6, False, "structured"), (1, 1536, 128, 128, 1e-5, True, "structured"),
    (2, 1000, 5120, 0, 1e-5, True, "structured"), (2, 100, 256, 256, 1e-6, False, "degenerate"),
    (3, 9, 512, 0, 1e-6, True, "structured"), (1, 1, 2560, 0, 1e-5, False, "iid"),
]


@pytest.mark.parametrize("B,HW,C0,C1,eps,silu,regime", APPLY_CASES)
def test_groupnorm_apply_paths(B, HW, C0, C1, eps, silu, regime):
    """groupnorm_silu, groupnorm_apply (statistics of each source) and groupnorm_apply_mr (float64 statistics rounded
    to fp32: the apply kernel alone) per (sample, group) against float64; the raw copy, groupnorm_silu against
    groupnorm_stats + groupnorm_apply, and two runs of the same call are bit-identical."""
    from adaprompt_b200 import ops
    C = C0 + C1
    x = nr.gn_input(regime, B, HW, C, seed=C + HW, device=DEV)
    x0, x1 = x[..., :C0].contiguous(), (x[..., C0:].contiguous() if C1 else None)
    gamma, beta = nr.affine(C, C, DEV)
    y_ref, mean, rstd = nr.gn_ref(x0, x1, gamma, beta, eps, silu)
    ys = {}
    raw = torch.empty(B, HW, C, dtype=torch.bfloat16, device=DEV)
    for run in range(2):
        ys[f"silu{run}"] = torch.empty(B, HW, C, dtype=torch.bfloat16, device=DEV)
        ops.groupnorm_silu(x0, gamma, beta, eps, silu, ys[f"silu{run}"], x1=x1, raw=raw if run else None)
    ys["apply"] = torch.empty(B, HW, C, dtype=torch.bfloat16, device=DEV)
    ops.groupnorm_apply(x0, ops.groupnorm_stats(x0), gamma, beta, eps, silu, ys["apply"], x1=x1,
                        st1=ops.groupnorm_stats(x1) if C1 else None)
    if not C1:
        ys["apply_mr"] = torch.empty(B, HW, C, dtype=torch.bfloat16, device=DEV)
        ops.groupnorm_apply_mr(x0, nr.stats_as_mr(mean, rstd), gamma, beta, silu, ys["apply_mr"])
    assert torch.equal(raw, x.to(torch.bfloat16))
    assert torch.equal(ys["silu0"], ys["silu1"])
    assert torch.equal(ys["silu0"], ys["apply"])
    lim = GN_OUT_GROUP
    if regime == "structured":
        _sens_check(f"apply {B} {HW} {C0}|{C1}", lim,
                    nr.gn_output_sensitivity(x, gamma, beta, eps, silu, _default_slots(B, HW)))
    for k, y in ys.items():
        wg, rel = nr.worst_group(y, y_ref), nr.rel_l2(y, y_ref)
        _seen(f"gn_out_group[{regime}]", wg)
        _seen("gn_out_rel", rel)
        assert wg < lim and rel < GN_OUT_REL, (k, wg, rel)


# ------------------------------------------------------------------------------------------------ GroupNorm backward
def _gn_bwd_case(B, HW, C, silu, dres, regime, seed=0):
    from adaprompt_b200 import ops
    x = nr.gn_input(regime, B, HW, C, seed=seed + C, device=DEV)
    dy = nr.gn_input(regime, B, HW, C, seed=seed + C + 1, device=DEV).to(torch.bfloat16)
    r = (torch.randn(B, HW, C, generator=torch.Generator().manual_seed(seed)).to(DEV) if dres else None)
    gamma, beta = nr.affine(C, seed + 2, DEV)
    mean, rstd = nr.gn_stats_ref(x, 1e-5)
    mr = nr.stats_as_mr(mean, rstd)
    # the reference takes the statistics the kernel gets: float64 values rounded to fp32
    m32, r32 = mr.reshape(B, 32, 2).unbind(-1)
    dx = ops.groupnorm_bwd(x, mr, gamma, beta, silu, dy, r)
    ref = nr.gn_bwd_ref(x, m32, r32, gamma, beta, silu, dy, r)
    label = f"gn bwd B={B} HW={HW} C={C} silu={silu} dres={dres} {regime}"
    wg = _seen("gn_bwd_group", nr.worst_group(dx, ref))
    if regime == "structured" and not dres:
        _sens_check(label, GN_BWD_GROUP, nr.gn_bwd_sensitivity(x, m32, r32, gamma, beta, silu, dy, _bwd_chunks(B, HW)))
    assert wg < GN_BWD_GROUP, (label, wg)
    if not dres:
        g = dx.double().reshape(B, HW, 32, C // 32)
        inv = _seen("gn_bwd_sum", (g.sum(dim=(1, 3)).abs() / g.abs().sum(dim=(1, 3)).clamp_min(1e-300)).max().item())
        assert inv < GN_BWD_SUM, (label, inv)
    assert torch.equal(dx, ops.groupnorm_bwd(x, mr, gamma, beta, silu, dy, r)), label


@pytest.mark.parametrize("C", [128, 256, 512, 320, 640, 960, 1280, 1920])
@pytest.mark.parametrize("HW,B", [(9, 2), (100, 16), (1000, 1), (4096, 2)])
def test_groupnorm_backward_direct(C, HW, B):
    """ops.groupnorm_bwd with the reference statistics: one chunk (HW = 9), uneven chunks (HW = 100 at B = 16: 6 chunks
    of 17 rows, the last 15; HW = 1000 at B = 1: 62 chunks of 17, the last three empty) and 256 chunks of 16 rows."""
    for silu, dres in ((True, False), (False, True)):
        _gn_bwd_case(B, HW, C, silu, dres, "structured")
    _gn_bwd_case(B, HW, C, True, True, "iid", seed=7)


def test_groupnorm_backward_wide_channels_after_narrow():
    """C = 2560 and 5120 need more than 48 KB of dynamic shared memory in gn_bwd_apply_kernel; run them after a
    narrower call in the same process, then the narrower one again."""
    for C, HW, B in ((640, 100, 2), (2560, 1000, 2), (5120, 100, 1), (2560, 9, 16), (5120, 1000, 1), (640, 100, 2)):
        for silu, dres in ((True, False), (False, True), (False, False)):
            _gn_bwd_case(B, HW, C, silu, dres, "structured", seed=C + HW)


@pytest.mark.parametrize("B,HW,C,silu", [(2, 256, 320, True), (1, 1000, 1280, False), (16, 64, 640, True)])
def test_groupnorm_fn_against_float64(B, HW, C, silu):
    """GroupNormFn forward and backward (kernel statistics throughout) against the float64 reference of the same op."""
    from adaprompt_b200.train import GroupNormFn
    x = nr.gn_input("structured", B, HW, C, seed=C, device=DEV).requires_grad_(True)
    gamma, beta = nr.affine(C, 3, DEV)
    dy = nr.gn_input("iid", B, HW, C, seed=C + 1, device=DEV).to(torch.bfloat16)
    y = GroupNormFn.apply(x, gamma, beta, 1e-5, silu)
    y.backward(dy)
    y_ref, mean, rstd = nr.gn_ref(x.detach(), None, gamma, beta, 1e-5, silu)
    ref = nr.gn_bwd_ref(x.detach(), mean, rstd, gamma, beta, silu, dy)
    wy = _seen("gn_out_group[structured]", nr.worst_group(y, y_ref))
    wd = _seen("gn_fn_group", nr.worst_group(x.grad, ref))
    assert wy < GN_OUT_GROUP and wd < GN_FN_GROUP, (wy, wd)


# ------------------------------------------------------------------------------------------------ LayerNorm
LN_ROWS = (1, 7, 9, 77, 4099)


@pytest.mark.parametrize("C", [4, 128, 384, 388, 640, 644, 768, 1280, 1284, 2048])
@pytest.mark.parametrize("out_dtype", [torch.bfloat16, torch.float32])
def test_layernorm_forward(C, out_dtype):
    """Both sides of every instantiation threshold (C / 4 float4 vectors per row: MAXV 3 up to 96, 5 up to 160,
    10 up to 320, 16 up to 512), rows not a multiple of the 8 rows of a block; per-row limits.  The kernel is
    two-pass, so the offset regime holds up to mean/std = 1000."""
    from adaprompt_b200 import ops
    gamma, beta = nr.affine(C, C, DEV)
    f32 = out_dtype == torch.float32
    for rows in LN_ROWS:
        for regime in ("iid", "structured", "offset30", "offset1000"):
            x = nr.ln_input(regime, rows, C, seed=rows + C, device=DEV)
            y = torch.full((rows, C), float("nan"), dtype=out_dtype, device=DEV)
            ops.layernorm(x, gamma, beta, 1e-5, y)
            ref = nr.ln_ref(x, gamma, beta, 1e-5)[0]
            wr = nr.worst_row(y, ref)
            if f32:
                lim = LN_F32_ROW_OFFSET if regime.startswith("offset") else LN_F32_ROW
                _seen(f"ln_f32_row[{'offset' if regime.startswith('offset') else 'iid'}]", wr)
            else:
                lim = LN_BF16_ROW
                _seen("ln_bf16_row", wr)
            if regime == "structured" and f32:
                _sens_check(f"ln C={C} rows={rows}", lim, nr.ln_sensitivity(x, gamma, beta, 1e-5))
            assert wr < lim, (C, rows, regime, out_dtype, wr)


@pytest.mark.parametrize("C", [2052, 130, 2])
def test_layernorm_rejects_unsupported_widths(C):
    """More than 2048 channels, or C % 4 != 0: ValueError from both directions, and no kernel runs."""
    from adaprompt_b200 import ops
    x = torch.zeros(8, C, device=DEV)
    g = torch.ones(C, device=DEV)
    torch.cuda.synchronize()
    with _kernels() as names:
        with pytest.raises(ValueError):
            ops.layernorm(x, g, g, 1e-5, torch.empty(8, C, dtype=torch.bfloat16, device=DEV))
        with pytest.raises(ValueError):
            ops.layernorm(x, g, g, 1e-5, torch.empty(8, C, device=DEV))
        with pytest.raises(ValueError):
            ops.layernorm_bwd(x, g, 1e-5, torch.zeros(8, C, device=DEV))
    assert not any("layernorm" in n for n in names), names


@pytest.mark.parametrize("C", [128, 384, 388, 768, 772, 1280, 1284, 2048])
@pytest.mark.parametrize("dy_dtype", [torch.bfloat16, torch.float32])
def test_layernorm_backward(C, dy_dtype):
    """MAXV 3 / 6 / 10 / 16 on both sides of each threshold, dy bf16 / fp32, dres on / off, dgamma / dbeta on / off.
    dx per row and bit-reproducible; dgamma / dbeta (fp32 atomics, accumulated into what the buffers hold) by rel-L2."""
    from adaprompt_b200 import ops
    gamma, _ = nr.affine(C, C + 1, DEV)
    for rows in LN_ROWS:
        x = nr.ln_input("structured", rows, C, seed=rows + C, device=DEV)
        dy = nr.ln_input("structured", rows, C, seed=rows + C + 1, device=DEV).to(dy_dtype)
        r = torch.randn(rows, C, generator=torch.Generator().manual_seed(rows)).to(DEV)
        _sens_check(f"ln bwd C={C} rows={rows}", LN_BWD_ROW, nr.ln_bwd_sensitivity(x, gamma, 1e-5, dy))
        for dres in (False, True):
            for params in (False, True):
                dg0 = torch.linspace(-1, 1, C, device=DEV) if params else None
                db0 = torch.linspace(2, -2, C, device=DEV) if params else None
                dg, db = (dg0.clone(), db0.clone()) if params else (None, None)
                dx = ops.layernorm_bwd(x, gamma, 1e-5, dy, r if dres else None, dg, db)
                ref, rg, rb = nr.ln_bwd_ref(x, gamma, 1e-5, dy, r if dres else None)
                wr = _seen("ln_bwd_row", nr.worst_row(dx, ref))
                assert wr < LN_BWD_ROW, (C, rows, dres, params, wr)
                if params:
                    eg = _seen("ln_param_rel", nr.rel_l2(dg - dg0, rg))
                    eb = _seen("ln_param_rel", nr.rel_l2(db - db0, rb))
                    assert eg < LN_PARAM_REL and eb < LN_PARAM_REL, (C, rows, eg, eb)
                if not dres:
                    s = _seen("ln_bwd_sum", (dx.double().sum(-1).abs() / dx.double().abs().sum(-1).clamp_min(1e-300))
                              .max().item())
                    assert s < LN_BWD_SUM, (C, rows, s)
                assert torch.equal(dx, ops.layernorm_bwd(x, gamma, 1e-5, dy, r if dres else None)), (C, rows)


# ------------------------------------------------------------------------------------------------ dispatch
def test_norm_dispatch_runs_every_kernel():
    """Each LayerNorm instantiation (4 widths x bf16 / fp32 output forward, 4 widths x bf16 / fp32 dy backward) and
    each GroupNorm kernel runs: a moved threshold cannot silently leave one untested."""
    from adaprompt_b200 import ops
    with _kernels() as names:
        for C in (384, 640, 1280, 2048):
            x = torch.randn(9, C, device=DEV)
            g = torch.ones(C, device=DEV)
            for dt in (torch.bfloat16, torch.float32):
                ops.layernorm(x, g, g, 1e-5, torch.empty(9, C, dtype=dt, device=DEV))
        for C in (384, 768, 1280, 2048):
            x = torch.randn(9, C, device=DEV)
            g = torch.ones(C, device=DEV)
            for dt in (torch.bfloat16, torch.float32):
                ops.layernorm_bwd(x, g, 1e-5, torch.randn(9, C, device=DEV).to(dt))
        x = torch.randn(2, 100, 320, device=DEV)
        g = torch.ones(320, device=DEV)
        y = torch.empty(2, 100, 320, dtype=torch.bfloat16, device=DEV)
        ops.groupnorm_silu(x, g, g, 1e-5, True, y)
        ops.groupnorm_bwd(x, ops.groupnorm_mean_rstd(x, ops.groupnorm_stats(x), 1e-5), g, g, True, y)
    want = [f"layernorm_kernel<{m},{f}>" for m in (3, 5, 10, 16) for f in ("false", "true")]
    want += [f"layernorm_bwd_kernel<{m},{f}>" for m in (3, 6, 10, 16) for f in ("false", "true")]
    want += ["gn_stats_kernel", "gn_finalize_kernel", "gn_apply_kernel", "gn_bwd_partial_kernel",
             "gn_bwd_finalize_kernel", "gn_bwd_apply_kernel"]
    missing = [w for w in want if not any(w in n for n in names)]
    assert not missing, (missing, sorted(n for n in names if "norm" in n or "gn_" in n))


# ------------------------------------------------------------------------------------------------ elementwise kernels
def _bf16_ulp(v):
    """One bf16 ulp at |v| (8 significant bits), float64."""
    a = v.abs().clamp_min(2.0 ** -126)
    return torch.exp2(torch.floor(torch.log2(a)) - 7)


def _gates(n, gen):
    """Gate / argument values: the erf and sigmoid tails up to |g| = 10, and a dense band around -0.75, where the
    derivatives of GELU and quick_gelu cross zero."""
    g = torch.cat([torch.linspace(-10, 10, n // 3), -0.75 + 0.05 * torch.randn(n // 3, generator=gen),
                   2 * torch.randn(n - 2 * (n // 3), generator=gen)])
    return g[torch.randperm(n, generator=gen)]


@pytest.mark.parametrize("T,F", [(37, 300), (5, 1280), (77, 20)])
def test_geglu_forward_backward_within_one_ulp(T, F):
    """h = a * gelu(g) and its gradients, each within 1 bf16 ulp of float64 of the exact bf16 inputs, plus an absolute
    slack of 2^-20 |dh| (|a| + |g| + 1): fp32 erf and exp carry absolute errors that matter only where the result
    cancels (d/dg near g = -0.75) or underflows (the erf tails)."""
    from adaprompt_b200 import ops
    gen = torch.Generator().manual_seed(T * F)
    a = torch.randn(T, F, generator=gen)
    g = _gates(T * F, gen).reshape(T, F)
    proj = torch.cat([a, g], 1).to(torch.bfloat16).to(DEV)
    dh = torch.randn(T, F, generator=gen).to(torch.bfloat16).to(DEV)
    h = ops.geglu_fwd(proj)
    dproj = ops.geglu_bwd(proj, dh)
    ad, gd, dd = proj[:, :F].double(), proj[:, F:].double(), dh.double()
    cdf = 0.5 * (1 + torch.erf(gd / 2 ** 0.5))
    pdf = torch.exp(-0.5 * gd * gd) / (2 * torch.pi) ** 0.5
    refs = {"h": (h, ad * gd * cdf, ad.abs() + gd.abs() + 1),
            "da": (dproj[:, :F], dd * gd * cdf, dd.abs() * (gd.abs() + 1)),
            "dg": (dproj[:, F:], dd * ad * (cdf + gd * pdf), dd.abs() * (ad.abs() + gd.abs() + 1))}
    for k, (got, ref, scale) in refs.items():
        excess = ((got.double() - ref).abs() - _bf16_ulp(ref) - 2.0 ** -20 * scale).max().item()
        assert excess <= 0, (k, excess)


@pytest.mark.parametrize("n", [77 * 3072 + 5, 1000])
def test_quick_gelu_forward_backward_within_one_ulp(n):
    from adaprompt_b200 import ops
    gen = torch.Generator().manual_seed(n)
    x = _gates(n, gen).to(torch.bfloat16).to(DEV)
    dy = torch.randn(n, generator=gen).to(torch.bfloat16).to(DEV)
    y, dx = ops.quick_gelu(x), ops.quick_gelu(x, dy)
    xd, dd = x.double(), dy.double()
    s = torch.sigmoid(1.702 * xd)
    for k, got, ref, scale in (("y", y, xd * s, xd.abs() + 1),
                               ("dx", dx, dd * s * (1 + 1.702 * xd * (1 - s)), dd.abs() * (xd.abs() + 1))):
        excess = ((got.double() - ref).abs() - _bf16_ulp(ref) - 2.0 ** -20 * scale).max().item()
        assert excess <= 0, (k, excess)


@pytest.mark.parametrize("B,H,W,C", [(2, 5, 3, 37), (1, 32, 32, 320), (3, 1, 1, 4)])
def test_sumpool2x2_and_zero_insert2x_bit_exact(B, H, W, C):
    from adaprompt_b200 import ops
    gen = torch.Generator().manual_seed(C)
    x = (torch.randn(B, 2 * H, 2 * W, C, generator=gen) * 3).to(DEV)
    ref = (x[:, 0::2, 0::2] + x[:, 0::2, 1::2]) + (x[:, 1::2, 0::2] + x[:, 1::2, 1::2])
    assert torch.equal(ops.sumpool2x2(x), ref)
    s = x[:, :H, :W].contiguous()
    z = ops.zero_insert2x(s)
    ref = torch.zeros(B, 2 * H, 2 * W, C, dtype=torch.bfloat16, device=DEV)
    ref[:, 0::2, 0::2] = s.to(torch.bfloat16)
    assert torch.equal(z, ref)


@pytest.mark.parametrize("R,C,ldo", [(45, 70, 56), (32, 32, 32), (1, 33, 9), (100, 3, 104)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_transpose_to_bf16_bit_exact(R, C, ldo, dtype):
    """out [C][ldo] = in^T rounded to bf16, pad columns R..ldo-1 zero, nothing written past C * ldo."""
    from adaprompt_b200 import _lib
    from adaprompt_b200._lib import AF_DTYPE_BF16, AF_DTYPE_F32
    lib = _lib.load()
    x = torch.randn(R, C, generator=torch.Generator().manual_seed(R * C)).to(dtype).to(DEV)
    sentinel = torch.tensor(-12345.0, dtype=torch.bfloat16)
    out = torch.full((C * ldo + 64,), sentinel.item(), dtype=torch.bfloat16, device=DEV)
    rc = lib.af_transpose_to_bf16(x.data_ptr(), AF_DTYPE_F32 if dtype == torch.float32 else AF_DTYPE_BF16, R, C, ldo,
                                  out.data_ptr(), _stream())
    assert rc == 0
    o = out[:C * ldo].reshape(C, ldo)
    assert torch.equal(o[:, :R], x.t().to(torch.bfloat16))
    assert torch.equal(o[:, R:], torch.zeros(C, ldo - R, dtype=torch.bfloat16, device=DEV))
    assert torch.all(out[C * ldo:] == sentinel.item())
