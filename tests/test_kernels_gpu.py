"""Per-kernel parity on a B200: every af_* entry point against a plain PyTorch fp32 reference of the same
op, on bf16-rounded operands (so only accumulation order / the documented bf16 roundings differ).
All calls go through the C ABI (adaprompt_b200.ops -> ctypes -> libadaface_b200.so)."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DEV = "cuda"


def _rel(a, b):
    a, b = a.float(), b.float()
    return ((a - b).norm() / b.norm().clamp_min(1e-12)).item()


def _rand(*shape, seed=0, scale=1.0, dtype=torch.float32):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(dtype).to(DEV)


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False


# ------------------------------------------------------------------------------------------------ GEMM
@pytest.mark.parametrize("M,N,K,bn", [
    (128, 128, 64, 0), (128, 64, 64, 64), (256, 320, 320, 0), (4096, 320, 320, 160), (1000, 640, 2560, 0),
    (77 * 3, 1280, 768, 0), (8192, 2560, 320, 256), (300, 256, 1280, 128), (64, 768, 320, 128), (512, 1280, 5120, 0),
])
def test_gemm_plain(M, N, K, bn):
    from adaprompt_b200 import ops
    a = _rand(M, K, seed=1, dtype=torch.bfloat16)
    w = _rand(N, K, seed=2, scale=K ** -0.5, dtype=torch.bfloat16)
    bias = _rand(N, seed=3)
    out = torch.empty(M, N, device=DEV, dtype=torch.float32)
    ops.gemm(a, w, out, bias=bias, bn=bn)
    ref = a.float() @ w.float().t() + bias
    assert _rel(out, ref) < 2e-5
    outb = torch.empty(M, N, device=DEV, dtype=torch.bfloat16)
    ops.gemm(a, w, outb, bias=bias, bn=bn)
    assert _rel(outb, ref) < 4e-3


def test_gemm_residual_rowbias_slice():
    from adaprompt_b200 import ops
    B, HW, N, K = 3, 256, 320, 640
    M = B * HW
    a = _rand(M, K, seed=1, dtype=torch.bfloat16)
    w = _rand(N, K, seed=2, scale=K ** -0.5, dtype=torch.bfloat16)
    bias = _rand(N, seed=3)
    rowbias = _rand(B, N, seed=4)
    res = _rand(M, N, seed=5)
    out = torch.zeros(M, 2 * N, device=DEV, dtype=torch.float32)
    ops.gemm(a, w, out[:, N:], bias=bias, rowbias=rowbias, rows_per_group=HW, residual=res, ldo=2 * N, ldr=N)
    ref = a.float() @ w.float().t() + bias + rowbias.repeat_interleave(HW, 0) + res
    assert _rel(out[:, N:], ref) < 2e-5
    assert out[:, :N].abs().max().item() == 0.0


def test_gemm_dual_source():
    from adaprompt_b200 import ops
    M, N, K0, K1 = 1024, 320, 640, 320
    a0 = _rand(M, K0, seed=1, dtype=torch.bfloat16)
    a1 = _rand(M, K1, seed=2, dtype=torch.bfloat16)
    w = _rand(N, K0 + K1, seed=3, scale=(K0 + K1) ** -0.5, dtype=torch.bfloat16)
    out = torch.empty(M, N, device=DEV, dtype=torch.float32)
    ops.gemm(a0, w, out, a1=a1)
    ref = torch.cat([a0, a1], 1).float() @ w.float().t()
    assert _rel(out, ref) < 2e-5


def test_gemm_geglu():
    from adaprompt_b200 import ops
    from adaprompt_b200.packing import pack_geglu
    M, C = 1024, 320
    x = _rand(M, C, seed=1, dtype=torch.bfloat16)
    w = _rand(8 * C, C, seed=2, scale=C ** -0.5)      # nn.Linear(C, 8C): rows [value 4C | gate 4C]
    b = _rand(8 * C, seed=3, scale=0.1)
    wp, bp = pack_geglu(w, b)
    out = torch.empty(M, 4 * C, device=DEV, dtype=torch.bfloat16)
    ops.gemm(x, wp.to(torch.bfloat16).contiguous(), out, bias=bp.contiguous(), geglu=True)
    h = x.float() @ w.to(torch.bfloat16).float().t() + b
    val, gate = h.chunk(2, dim=-1)
    ref = val * F.gelu(gate)
    assert _rel(out, ref) < 4e-3


def test_gemm_swap_ab_transposed_out():
    """V^T = Wv . X^T : the same kernel with the weight as the M operand."""
    from adaprompt_b200 import ops
    tokens, C, K = 2048, 320, 320
    x = _rand(tokens, K, seed=1, dtype=torch.bfloat16)
    wv = _rand(C, K, seed=2, scale=K ** -0.5, dtype=torch.bfloat16)
    vt = torch.empty(C, tokens, device=DEV, dtype=torch.bfloat16)
    ops.gemm(wv, x, vt, bn=128)
    ref = (x.float() @ wv.float().t()).t()
    assert _rel(vt, ref) < 4e-3


# ------------------------------------------------------------------------------------------------ conv3x3
def _conv_ref(x_nhwc, w_oihw, bias, stride):
    y = F.conv2d(x_nhwc.float().permute(0, 3, 1, 2), w_oihw.float(), bias, stride=stride, padding=1)
    return y.permute(0, 2, 3, 1).contiguous()


@pytest.mark.parametrize("B,H,W,Cin,Cout,stride", [
    (2, 64, 64, 320, 320, 1), (2, 32, 32, 640, 640, 1), (2, 16, 16, 1280, 1280, 1), (3, 8, 8, 1280, 1280, 1),
    (1, 64, 64, 320, 320, 2), (2, 32, 32, 640, 640, 2), (3, 16, 16, 1280, 1280, 2),
    (1, 96, 96, 320, 320, 1), (1, 24, 24, 640, 320, 1), (2, 12, 12, 1280, 640, 1),
])
def test_conv3x3(B, H, W, Cin, Cout, stride):
    from adaprompt_b200 import ops
    from adaprompt_b200.packing import pack_conv3x3
    x = _rand(B, H, W, Cin, seed=1, dtype=torch.bfloat16)
    w = _rand(Cout, Cin, 3, 3, seed=2, scale=(9 * Cin) ** -0.5).to(torch.bfloat16)
    bias = _rand(Cout, seed=3)
    Ho, Wo = H // stride, W // stride
    out = torch.empty(B, Ho, Wo, Cout, device=DEV, dtype=torch.float32)
    ops.conv3x3(x, pack_conv3x3(w), out, stride=stride, bias=bias)
    ref = _conv_ref(x, w, bias, stride)
    assert _rel(out, ref) < 2e-5


def test_conv3x3_dual_source_rowbias_residual():
    from adaprompt_b200 import ops
    from adaprompt_b200.packing import pack_conv3x3
    B, H, W, C0, C1, Cout = 2, 32, 32, 640, 320, 640
    x0 = _rand(B, H, W, C0, seed=1, dtype=torch.bfloat16)
    x1 = _rand(B, H, W, C1, seed=2, dtype=torch.bfloat16)
    w = _rand(Cout, C0 + C1, 3, 3, seed=3, scale=(9 * (C0 + C1)) ** -0.5).to(torch.bfloat16)
    bias = _rand(Cout, seed=4)
    emb = _rand(B, Cout, seed=5)
    res = _rand(B, H, W, Cout, seed=6)
    out = torch.empty(B, H, W, Cout, device=DEV, dtype=torch.float32)
    ops.conv3x3(x0, pack_conv3x3(w), out, x1=x1, bias=bias, rowbias=emb, residual=res)
    ref = _conv_ref(torch.cat([x0, x1], -1), w, bias, 1) + emb[:, None, None, :] + res
    assert _rel(out, ref) < 2e-5


# ------------------------------------------------------------------------------------------------ attention
ATTN_ROW_TOL = 1e-2       # worst rel-L2 over (sample, head, query row); 4.5e-3 seen on a B200
# |lse - ref| in log2 units.  The tile kernels sum l from the bf16-rounded P, whose relative error is up to 2^-8; a row
# dominated by one key (large scores) reaches log2(1 + 2^-8) = 5.62e-3 (seen: 5.63e-3, 2.3e-3 without dominant keys)
ATTN_LSE_TOL = 6e-3
POISON = 2.0 ** 127       # finite and exact in bf16; 0 * POISON = 0 where the kernels give a key exactly zero weight


def _attn_ref(qs, kb, vb, km=None):
    """af_attention_bf16 in float64 (attention.py:198-242) on the kernel's bf16 operands; CPU or CUDA tensors.
    qs [B, Nq, h, d] carries d^-1/2 * log2(e), so the scores s are in the exp2 domain; kb, vb [B, Nk, h, d]; km [B, Nk]
    (nonzero = attend) or None.  Masked scores are filled with -finfo.max as in the reference, so a sample that attends
    to no key gets a uniform softmax.  -> (O [B, Nq, h*d], lse [B, h, Nq] = log2 sum_j 2^s_j over the attended keys, +inf
    where there are none)."""
    B, Nq, h, d = qs.shape
    s = torch.einsum("bihd,bjhd->bhij", qs.double(), kb.double())
    keep = torch.ones(B, kb.shape[1], dtype=torch.bool, device=s.device) if km is None else km.bool()
    keep = keep[:, None, None, :]
    p = torch.softmax(s.masked_fill(~keep, -torch.finfo(torch.float64).max) * math.log(2.0), dim=-1)
    o = torch.einsum("bhij,bjhd->bihd", p, vb.double()).reshape(B, Nq, h * d)
    lse = torch.logsumexp(s.masked_fill(~keep, float("-inf")) * math.log(2.0), dim=-1) / math.log(2.0)
    return o, lse.masked_fill(torch.isneginf(lse), float("inf"))


def _attn_errors(out, lse, ref, ref_lse):
    """Global rel-L2 of O, the worst rel-L2 over (sample, head, query row) and the worst |lse - ref|.  Rows whose
    reference lse is +inf must be +inf in lse too (a non-finite difference otherwise)."""
    B, Nq, C = ref.shape
    heads = lse.shape[1]
    diff = out.double() - ref
    rows = diff.view(B, Nq, heads, -1).norm(dim=-1) / ref.view(B, Nq, heads, -1).norm(dim=-1).clamp_min(1e-30)
    inf = torch.isinf(ref_lse)
    lse_d = lse.double()
    lse_err = torch.where(inf, torch.where(lse_d == ref_lse, 0.0, float("inf")), (lse_d - ref_lse).abs())
    return {"rel": (diff.norm() / ref.norm()).item(), "row": rows.max().item(), "lse": lse_err.max().item()}


def _attn_case(B, N, Nk, d, seed=0, mask=False, cross=False, boost=None, poison=False, empty=None, tol=6e-3):
    """Runs ops.attention_lse and ops.attention on one problem: the two O must be bit-identical, and O / lse must match
    _attn_ref (global rel-L2 < tol, worst row < ATTN_ROW_TOL, lse < ATTN_LSE_TOL).
    cross: keys stored with a sample stride padded to a multiple of 8 (the cached-context layout).
    mask: random key mask that keeps key 0; empty: index of a sample whose mask keeps no key.
    boost = (first_key, factor): keys from first_key on are scaled, so that scores far above the first block's appear
    late in the key loop (the lazy-reference / overflow paths of the attention kernels).
    poison: the V^T columns that must get zero weight hold +-2^127 - masked keys of samples that attend to some key,
    [Nk, kv_stride) of every sample and [B*kv_stride, ldvt) - and masked keys' K rows are scaled by 2^10 (a maximum taken
    before masking would see them).  Returns the errors."""
    heads = 8
    C = heads * d
    dp = 48 if d == 40 else d
    scale = d ** -0.5
    q = _rand(B, N, heads, d, seed=seed + 1)
    k = _rand(B, Nk, heads, d, seed=seed + 2)
    v = _rand(B, Nk, heads, d, seed=seed + 3)
    if boost is not None:
        k[:, boost[0]:] *= boost[1]
    qs = (q * (scale * math.log2(math.e))).to(torch.bfloat16)
    kb, vb = k.to(torch.bfloat16), v.to(torch.bfloat16)
    km = None
    if mask or empty is not None:
        g = torch.Generator().manual_seed(seed + 9)
        km = (torch.rand(B, Nk, generator=g) > 0.3).to(torch.uint8).to(DEV)
        km[:, 0] = 1
        if empty is not None:
            km[empty] = 0
    ref, ref_lse = _attn_ref(qs, kb, vb, km)

    qbuf = torch.zeros(B, N, heads, dp, device=DEV, dtype=torch.bfloat16)
    nk_pad = ((Nk + 7) // 8) * 8 if cross else Nk
    ldvt = (max(64, B * nk_pad) + 7) // 8 * 8 + (64 if poison else 0)     # a multiple of 8 (16-byte TMA rows)
    kbuf = torch.zeros(B, nk_pad, heads, dp, device=DEV, dtype=torch.bfloat16)
    qbuf[..., :d] = qs
    kbuf[:, :Nk, :, :d] = kb
    vt = torch.zeros(C, ldvt, device=DEV, dtype=torch.bfloat16)
    vt3 = vt[:, :B * nk_pad].view(C, B, nk_pad)
    vt3[:, :, :Nk] = vb.permute(2, 3, 0, 1).reshape(C, B, Nk)
    if poison:
        g = torch.Generator().manual_seed(seed + 10)

        def big(*shape):
            return ((torch.randint(0, 2, shape, generator=g) * 2 - 1) * POISON).to(torch.bfloat16).to(DEV)

        vt3[:, :, Nk:] = big(C, B, nk_pad - Nk)
        vt[:, B * nk_pad:] = big(C, ldvt - B * nk_pad)
        if km is not None:
            dead = (km == 0) & (km.sum(1, keepdim=True) > 0)
            vt3[:, :, :Nk] = torch.where(dead[None], big(C, B, Nk), vt3[:, :, :Nk])
            kv = kbuf[:, :Nk]
            kv[km == 0] = kv[km == 0] * 1024.0

    return _attn_check(qbuf, kbuf, vt, ref, ref_lse, tol, dict(
        B=B, heads=heads, Nq=N, Nk=Nk, d=d, ldq=heads * dp, ldk=heads * dp, ldvt=ldvt, kv_stride=nk_pad, key_mask=km),
        f"mask={mask} cross={cross} boost={boost} poison={poison} empty={empty}")


def _attn_check(q, k, vt, ref, ref_lse, tol, args, label=""):
    """ops.attention_lse and ops.attention on the same operands (args: their keyword arguments): the two O must be
    bit-identical, and O / lse must match the reference (global rel-L2 < tol, worst row < ATTN_ROW_TOL, lse <
    ATTN_LSE_TOL).  Prints the errors and returns them."""
    from adaprompt_b200 import ops
    B, Nq, heads = args["B"], args["Nq"], args["heads"]
    out = torch.full((B, Nq, ref.shape[-1]), float("nan"), device=DEV, dtype=torch.bfloat16)
    out2 = torch.full_like(out, float("nan"))
    lse = torch.full((B, heads, Nq), float("nan"), device=DEV)
    ops.attention_lse(q, k, vt, out, lse, **args)
    ops.attention(q, k, vt, out2, **args)
    assert torch.equal(out, out2), "attention and attention_lse disagree"
    e = _attn_errors(out, lse, ref, ref_lse)
    print(f"\nattention B={B} Nq={Nq} Nk={args['Nk']} d={args['d']} {label}: rel {e['rel']:.2e}  "
          f"worst row {e['row']:.2e}  lse {e['lse']:.2e}")
    assert e["rel"] < tol and e["row"] < ATTN_ROW_TOL and e["lse"] < ATTN_LSE_TOL, e
    return e


@pytest.mark.parametrize("B,N,d", [(1, 4096, 40), (2, 1024, 80), (2, 256, 160), (3, 64, 160), (1, 2304, 80),
                                   (2, 144, 160), (1, 576, 160),
                                   (3, 296, 40),       # ragged last key block: masked tile kernel, d = 40
                                   (2, 1600, 40),      # the 40x40 latent
                                   (2, 144, 80),       # the 12x12 map: masked tile kernel, d = 80
                                   (2, 64, 40)])       # generic kernel, d = 40
def test_self_attention(B, N, d):
    _attn_case(B, N, N, d)


@pytest.mark.parametrize("B,N,d,first,factor", [
    (1, 1024, 40, 640, 40.0),      # scores up to ~2^+-250 from key 640 on: P overflows on the unguarded fast path -> second pass
    (1, 1024, 40, 640, 14.0),      # ~2^90: no overflow of P, but beyond the 2^64 window
    (2, 1024, 80, 512, 30.0),      # d = 80 keeps the per-block guard
    (1, 4096, 40, 3968, 60.0),     # only the LAST key block is extreme
])
def test_self_attention_large_scores_late_in_the_key_loop(B, N, d, first, factor):
    """Rows whose maximum moves far away from the first block's: the result must be the exact softmax (no inf / NaN, no
    stale reference) whichever path the kernel takes to get there."""
    _attn_case(B, N, N, d, seed=11, boost=(first, factor), tol=8e-3)


@pytest.mark.parametrize("B,N,d", [(2, 4096, 40), (2, 1024, 80), (2, 256, 160), (2, 64, 160)])
def test_cross_attention_77(B, N, d):
    _attn_case(B, N, 77, d, seed=5, cross=True)


@pytest.mark.parametrize("B,N,d", [(2, 1024, 40), (2, 256, 80), (3, 64, 160), (2, 16, 160)])
def test_self_attention_fused_qk_buffer(B, N, d):
    """Layout the UNet uses: one [tokens, Q|K] buffer (K = column view), V^T [C, tokens]."""
    heads, C = 8, 8 * d
    dp = 48 if d == 40 else d
    q = _rand(B, N, heads, d, seed=11)
    k = _rand(B, N, heads, d, seed=12)
    v = _rand(B, N, heads, d, seed=13)
    qs = (q * (d ** -0.5 * math.log2(math.e))).to(torch.bfloat16)
    kb, vb = k.to(torch.bfloat16), v.to(torch.bfloat16)
    qk = torch.zeros(B * N, 2, heads, dp, device=DEV, dtype=torch.bfloat16)
    qk[:, 0, :, :d] = qs.reshape(B * N, heads, d)
    qk[:, 1, :, :d] = kb.reshape(B * N, heads, d)
    qk = qk.reshape(B * N, 2 * heads * dp)
    ldvt = max(64, B * N)
    vt = torch.zeros(C, ldvt, device=DEV, dtype=torch.bfloat16)
    vt[:, :B * N] = vb.permute(2, 3, 0, 1).reshape(C, B * N)
    ref, ref_lse = _attn_ref(qs, kb, vb)
    _attn_check(qk, qk[:, heads * dp:], vt, ref, ref_lse, 6e-3, dict(B=B, heads=heads, Nq=N, Nk=N, d=d,
                ldq=2 * heads * dp, ldk=2 * heads * dp, ldvt=ldvt, kv_stride=N), "fused [Q|K]")


def test_cross_attention_padded_kv_stride():
    """Cached-context layout: 77 keys stored with a sample stride of 80 rows (K) / columns (V^T)."""
    B, N, d, Nk, pad = 3, 256, 80, 77, 80
    heads, C = 8, 640
    q = _rand(B, N, heads, d, seed=21)
    k = _rand(B, Nk, heads, d, seed=22)
    v = _rand(B, Nk, heads, d, seed=23)
    qs = (q * (d ** -0.5 * math.log2(math.e))).to(torch.bfloat16)
    kb, vb = k.to(torch.bfloat16), v.to(torch.bfloat16)
    kbuf = torch.zeros(B, pad, C, device=DEV, dtype=torch.bfloat16)
    kbuf[:, :Nk] = kb.reshape(B, Nk, C)
    vt = torch.zeros(C, B, pad, device=DEV, dtype=torch.bfloat16)
    vt[:, :, :Nk] = vb.permute(2, 3, 0, 1).reshape(C, B, Nk)
    ref, ref_lse = _attn_ref(qs, kb, vb)
    _attn_check(qs.reshape(B * N, C).contiguous(), kbuf, vt, ref, ref_lse, 6e-3, dict(B=B, heads=heads, Nq=N, Nk=Nk,
                d=d, ldq=C, ldk=C, ldvt=B * pad, kv_stride=pad), "padded kv_stride")


def test_attention_rejects_unaligned_sample_stride():
    """2x2 feature maps (N = 4) with B > 1 would put V^T boxes on 8-byte boundaries: refused, not mis-run."""
    from adaprompt_b200 import ops
    t = torch.zeros(8, 2560, device=DEV, dtype=torch.bfloat16)
    vt = torch.zeros(1280, 64, device=DEV, dtype=torch.bfloat16)
    with pytest.raises(ValueError):
        ops.attention(t, t[:, 1280:], vt, torch.empty(8, 1280, device=DEV, dtype=torch.bfloat16), B=2, heads=8, Nq=4,
                      Nk=4, d=160, ldq=2560, ldk=2560, ldvt=64, kv_stride=4)


def test_self_attention_key_mask():
    _attn_case(2, 1024, 1024, 80, seed=7, mask=True)


@pytest.mark.parametrize("B,N,Nk,d,mask", [(2, 2304, 77, 80, False), (1, 9216, 77, 40, False), (3, 300, 77, 40, True),
                                           (2, 1024, 128, 80, True), (3, 512, 24, 40, False), (16, 4096, 77, 40, False),
                                           (5, 384, 100, 80, False),
                                           # 16-key chunks NCH = 1, 1, 2, 3, 4, 6 at both head dims
                                           (2, 300, 1, 40, False), (2, 256, 1, 80, True), (2, 300, 16, 40, True),
                                           (2, 384, 16, 80, False), (2, 300, 17, 40, False), (2, 256, 17, 80, True),
                                           (2, 300, 40, 40, True), (2, 640, 40, 80, False), (2, 256, 64, 40, False),
                                           (2, 300, 64, 80, True), (2, 300, 96, 40, True), (2, 256, 96, 80, False),
                                           (1, 256, 128, 40, False)])     # smallest query count that takes xattn
def test_short_context_attention(B, N, Nk, d, mask):
    """xattn.cu: K / V resident per (sample, head), ragged query tiles, key masks, every key-count class."""
    _attn_case(B, N, Nk, d, seed=31, mask=mask, cross=True)


# (B, Nq, Nk, d, mask, cross) -> the kernel af_attention_bf16 picks (attention.cu: attention_impl)
ATTN_MATRIX = [
    pytest.param(2, 1000, 1000, 40, True, False, id="tile40m-1000-mask"),
    pytest.param(1, 4096, 4096, 40, True, False, id="tile40m-4096-mask"),
    pytest.param(2, 300, 200, 40, False, True, id="tile40m-300x200-cross"),
    pytest.param(1, 256, 129, 40, False, False, id="tile40m-boundary-129"),
    pytest.param(2, 1000, 1000, 80, True, False, id="tile80m-1000-mask"),
    pytest.param(3, 600, 300, 80, True, True, id="tile80m-600x300-mask-cross"),
    pytest.param(1, 256, 129, 80, False, False, id="tile80m-boundary-129"),
    pytest.param(2, 300, 1024, 40, False, False, id="tile40-300x1024"),
    pytest.param(2, 200, 1024, 80, False, False, id="tile80-200x1024"),
    pytest.param(1, 255, 128, 40, False, False, id="generic40-boundary-255"),
    pytest.param(3, 200, 77, 40, True, True, id="generic40-200x77-mask"),
    pytest.param(2, 144, 77, 80, False, True, id="generic80-144x77"),
    pytest.param(2, 100, 100, 80, True, True, id="generic80-100-mask-cross"),
    pytest.param(2, 64, 64, 160, True, False, id="generic160-64-mask"),
    pytest.param(3, 96, 77, 160, True, True, id="generic160-96x77-mask"),
]


@pytest.mark.parametrize("B,Nq,Nk,d,mask,cross", ATTN_MATRIX)
def test_attention_dispatch_matrix(B, Nq, Nk, d, mask, cross):
    """Every kernel family and instantiation behind af_attention_bf16: key masks, ragged key and query tails, Nq != Nk,
    and the shapes on either side of each dispatch threshold."""
    _attn_case(B, Nq, Nk, d, seed=41, mask=mask, cross=cross)


@pytest.mark.parametrize("B,Nq,Nk,d,mask,cross", [
    pytest.param(2, 1000, 1000, 40, True, False, id="tile40m-mask"),
    pytest.param(3, 296, 296, 40, False, False, id="tile40m-ragged"),
    pytest.param(2, 300, 200, 40, True, True, id="tile40m-mask-cross"),
    pytest.param(2, 1000, 1000, 80, True, False, id="tile80m-mask"),
    pytest.param(3, 600, 300, 80, True, True, id="tile80m-mask-cross"),
    pytest.param(2, 144, 144, 80, False, False, id="tile80m-ragged"),
    pytest.param(3, 200, 77, 40, True, True, id="generic40-mask-cross"),
    pytest.param(2, 100, 100, 80, True, True, id="generic80-mask-cross"),
    pytest.param(3, 96, 77, 160, True, True, id="generic160-mask-cross"),
    pytest.param(2, 300, 77, 40, True, True, id="xattn40-mask-cross"),
    pytest.param(2, 256, 17, 80, True, True, id="xattn80-mask-cross"),
])
def test_attention_masked_keys_carry_no_weight(B, Nq, Nk, d, mask, cross):
    """Masked keys, keys past Nk and V^T columns past the last sample hold +-2^127 in V^T (and masked keys a K scaled by
    2^10): any nonzero weight on them shows up as a wrong output row."""
    _attn_case(B, Nq, Nk, d, seed=51, mask=mask, cross=cross, poison=True)


@pytest.mark.parametrize("B,Nq,Nk,d,cross,first,factor", [
    (2, 1000, 1000, 40, False, 640, 40.0),      # masked tile kernel: per-block guard and lazy reference
    (2, 1000, 1000, 80, False, 512, 30.0),
    (2, 100, 100, 80, True, 64, 30.0),          # generic kernel
])
def test_masked_attention_large_scores_late_in_the_key_loop(B, Nq, Nk, d, cross, first, factor):
    _attn_case(B, Nq, Nk, d, seed=13, mask=True, cross=cross, boost=(first, factor), tol=8e-3)


@pytest.mark.parametrize("B,Nq,Nk,d,cross,empty", [
    pytest.param(2, 300, 77, 40, True, 1, id="xattn40"),
    pytest.param(3, 1000, 1000, 40, False, 1, id="tile40m"),
    pytest.param(2, 1000, 1000, 80, False, 0, id="tile80m"),
    pytest.param(3, 200, 77, 40, True, 2, id="generic40"),
    pytest.param(2, 100, 100, 80, True, 1, id="generic80"),
    pytest.param(2, 64, 64, 160, False, 0, id="generic160"),
])
def test_attention_fully_masked_sample(B, Nq, Nk, d, cross, empty):
    """A sample whose key mask keeps no key: the reference's -finfo.max fill makes its softmax uniform, so each of its
    rows is the mean of V over its Nk keys and its lse is +inf; the other samples (partial masks) are unaffected."""
    _attn_case(B, Nq, Nk, d, seed=61, mask=True, cross=cross, empty=empty, poison=True)


def test_attention_dispatch_runs_every_kernel():
    """Each case of the dispatch matrix runs the kernel it is meant to: a moved threshold cannot silently leave an
    instantiation untested."""
    cases = [((2, 300, nk, d), dict(cross=True)) for d in (40, 80) for nk in (1, 17, 40, 64, 96)]
    cases += [((1, 256, 256, 40), {}), ((1, 256, 129, 40), {}), ((1, 256, 256, 80), {}), ((1, 256, 129, 80), {}),
              ((1, 255, 128, 40), {}), ((2, 144, 77, 80), dict(cross=True)), ((2, 64, 64, 160), dict(mask=True))]
    want = [f"xattn_kernel<{d},{n}>" for d in (40, 80) for n in (1, 2, 3, 4, 6)]
    want += ["attention_tile_kernel<40,3,false,false>", "attention_tile_kernel<40,0,true,false>",
             "attention_tile_kernel<80,0,false,false>", "attention_tile_kernel<80,0,true,false>",
             "attention_kernel<40>", "attention_kernel<80>", "attention_kernel<160>", "attention_empty_mask_kernel"]
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for shape, kw in cases:
            _attn_case(*shape, seed=71, **kw)
        torch.cuda.synchronize()
    names = {e.key.replace(" ", "") for e in prof.key_averages()}
    missing = [w for w in want if not any(w in n for n in names)]
    assert not missing, (missing, sorted(n for n in names if "attention" in n or "xattn" in n))


@pytest.mark.parametrize("d,N", [(40, 1000), (160, 64)])
def test_cross_attention_module_fully_masked_sample(d, N):
    """CrossAttention.forward(x, mask=...) as self-attention, sample 0 masked out entirely, sample 1 partially, against
    oracle.unet_oracle.cross_attention on the same weights."""
    from adaprompt_b200.attention import CrossAttention
    from oracle.unet_oracle import cross_attention
    C = 8 * d
    torch.manual_seed(3)
    attn = CrossAttention(C, heads=8, dim_head=d).to(DEV)
    x = _rand(2, N, C, seed=81)
    g = torch.Generator().manual_seed(82)
    mask = torch.rand(2, N, generator=g) > 0.5
    mask[0] = False
    with torch.no_grad():
        out = attn(x, mask=mask.to(DEV))
    sd = {f"a.{k}": v.detach().float().cpu() for k, v in attn.state_dict().items()}
    ref = cross_attention(sd, "a", x.cpu(), mask=mask)
    err = _rel(out.cpu(), ref)
    print(f"\nCrossAttention d={d} N={N} with a fully masked sample: rel {err:.2e}")
    assert err < 1e-2


# ------------------------------------------------------------------------------------------------ materialised scores
def _straddling_cols(M, nk):
    """M distinct key columns below nk, starting with those on either side of the 31|32 and 63|64 boundaries (the
    32-key lane groups of xattn_explicit)."""
    cand = [c for c in [31, 32, 63, 64] + list(range(nk)) if c < nk]
    return list(dict.fromkeys(cand))[:M]


@pytest.mark.parametrize("ks", [2, 3, 4])
@pytest.mark.parametrize("Hf,Wf", [(8, 8), (6, 10), (1, 7)])
def test_conv_attn_scores(ks, Hf, Wf):
    """ops.conv_attn_scores against oracle.unet_oracle.conv_attn_columns: sample 0 without the subject (cols = -1),
    sample 1 with columns across the 31|32 and 63|64 boundaries, sample 2 with random columns.  The oracle's restatement
    is pinned to the upstream replace_rows_by_conv_attn by a golden only at ks = 3; at ks = 2 and 4 (even kernels, uneven
    padding) it is checked against the restatement alone."""
    from adaprompt_b200 import ops
    from oracle.unet_oracle import conv_attn_columns
    B, heads, nk, M = 3, 8, 77, ks * ks
    N = Hf * Wf
    score = _rand(B, heads, N, nk, seed=91, scale=3.0)
    g = torch.Generator().manual_seed(92)
    cols = torch.stack([torch.full((M,), -1, dtype=torch.int64), torch.tensor(_straddling_cols(M, nk)),
                        torch.randperm(nk, generator=g)[:M]])
    ov = ops.conv_attn_scores(score, cols.to(torch.int32).to(DEV), B=B, heads=heads, Hf=Hf, Wf=Wf, nk=nk, ks=ks)
    ref = torch.zeros(B, heads, N, M, dtype=torch.float64)
    sc = score.double().cpu()
    for b in (1, 2):
        ref[b] = conv_attn_columns(sc[b], cols[b], (Hf, Wf), ks).permute(1, 2, 0)
    assert torch.equal(ov[0], torch.zeros_like(ov[0]))
    assert _rel(ov.cpu().double(), ref) < 1e-5


def _xattn_explicit_params():
    ps = []
    for d in (40, 80, 160):
        for nk in (1, 33, 77, 96):
            for N in (1, 64, 100):
                for ov in (False, True) if nk >= 18 else (False,):
                    ps.append(pytest.param(d, nk, N, ov, id=f"d{d}-nk{nk}-N{N}{'-override' if ov else ''}"))
    return ps


@pytest.mark.parametrize("d,nk,N,override", _xattn_explicit_params())
def test_xattn_explicit(d, nk, N, override):
    """ops.xattn_explicit against a float64 restatement of oracle.unet_oracle.cross_attention (sim, column replacement,
    softmax, attn.v, q * sqrt(scale)), two samples with the key stride padded to 8.  override: two subjects of ks = 3
    (n_ov = 18 columns) replace score columns, sample 0 has only the first, sample 1 only the second.  nk = 96 at d = 160 is
    the largest shared-memory configuration."""
    from adaprompt_b200 import ops
    B, heads = 2, 8
    C = heads * d
    dp = 48 if d == 40 else d
    kv_stride = (nk + 7) // 8 * 8
    scale = d ** -0.5
    qs = (_rand(B, N, heads, d, seed=101) * (scale * math.log2(math.e))).to(torch.bfloat16)
    kb = _rand(B, nk, heads, d, seed=102).to(torch.bfloat16)
    vb = _rand(B, nk, heads, d, seed=103).to(torch.bfloat16)
    qbuf = torch.zeros(B * N, heads, dp, device=DEV, dtype=torch.bfloat16)
    qbuf[:, :, :d] = qs.reshape(B * N, heads, d)
    kbuf = torch.zeros(B, kv_stride, heads, dp, device=DEV, dtype=torch.bfloat16)
    kbuf[:, :nk, :, :d] = kb
    kbuf[:, nk:, :, :d] = POISON           # padding keys are never read
    ldvt = max(64, B * kv_stride)
    vt = torch.full((C, ldvt), POISON, device=DEV, dtype=torch.bfloat16)
    vt[:, :B * kv_stride].view(C, B, kv_stride)[:, :, :nk] = vb.permute(2, 3, 0, 1).reshape(C, B, nk)
    ov = cols = None
    if override:
        M = 9
        ov = _rand(B, heads, N, 2 * M, seed=104, scale=2.0)
        c1, c2 = _straddling_cols(M, nk), list(range(nk - M, nk))[::-1]
        cols = torch.tensor([c1 + [-1] * M, [-1] * M + c2], dtype=torch.int32, device=DEV)
    r = ops.xattn_explicit(qbuf.reshape(B * N, heads * dp), kbuf.reshape(B * kv_stride, heads * dp), vt, B=B, heads=heads,
                           N=N, nk=nk, d=d, ldq=heads * dp, ldk=heads * dp, ldvt=ldvt, kv_stride=kv_stride, override=ov,
                           ov_cols=cols, want_out=True, want_scores=True, want_attn=True, want_q=True)
    # reference (oracle cross_attention :220-239): q = qs / (scale log2 e) is the unscaled query
    q = qs.double().permute(0, 2, 1, 3) / (scale * math.log2(math.e))
    sim = torch.einsum("bhid,bjhd->bhij", q, kb.double()) * scale
    if override:
        for b in range(B):
            for m in range(2 * M):
                c = int(cols[b, m])
                if c >= 0:
                    sim[b, :, :, c] = ov[b, :, :, m].double()
    attn = sim.softmax(dim=-1)
    out = torch.einsum("bhij,bjhd->bihd", attn, vb.double()).reshape(B * N, C)
    errs = {"attnscore": _rel(r["attnscore"].double(), sim), "attn": _rel(r["attn"].double(), attn),
            "q": _rel(r["q"].double(), q * scale ** 0.5), "out": _rel(r["out"].double(), out)}
    print(f"\nxattn_explicit d={d} nk={nk} N={N} override={override}: {errs}")
    assert errs["attnscore"] < 1e-5 and errs["attn"] < 1e-5 and errs["q"] < 1e-5 and errs["out"] < 6e-3, errs


# ------------------------------------------------------------------------------------------------ norms
@pytest.mark.parametrize("B,HW,C0,C1,eps,silu", [
    (2, 4096, 320, 0, 1e-5, True), (2, 1024, 640, 320, 1e-5, True), (3, 256, 1280, 640, 1e-5, True),
    (2, 64, 1280, 1280, 1e-5, True), (2, 4096, 320, 0, 1e-6, False), (1, 1024, 640, 640, 1e-5, True),
    (16, 64, 2560 - 1280, 1280, 1e-5, True),
])
def test_groupnorm_silu(B, HW, C0, C1, eps, silu):
    from adaprompt_b200 import ops
    x0 = _rand(B, HW, C0, seed=1) * 2 + 0.3
    x1 = _rand(B, HW, C1, seed=2) - 0.5 if C1 else None
    C = C0 + C1
    gamma = 1 + 0.1 * _rand(C, seed=3)
    beta = 0.1 * _rand(C, seed=4)
    out = torch.empty(B, HW, C, device=DEV, dtype=torch.bfloat16)
    raw = torch.empty(B, HW, C, device=DEV, dtype=torch.bfloat16)
    ops.groupnorm_silu(x0, gamma, beta, eps, silu, out, x1=x1, raw=raw)
    x = x0 if x1 is None else torch.cat([x0, x1], -1)
    ref = F.group_norm(x.permute(0, 2, 1), 32, gamma, beta, eps).permute(0, 2, 1)
    if silu:
        ref = F.silu(ref)
    assert _rel(out, ref) < 3e-3
    assert (out.float() - ref).abs().max().item() < 0.05
    assert torch.equal(raw, x.to(torch.bfloat16))


@pytest.mark.parametrize("rows,C", [(4096, 320), (2048, 640), (512, 1280), (77, 768), (33, 1024)])
def test_layernorm(rows, C):
    from adaprompt_b200 import ops
    x = _rand(rows, C, seed=1) * 1.7 + 0.2
    gamma = 1 + 0.1 * _rand(C, seed=2)
    beta = 0.1 * _rand(C, seed=3)
    out = torch.empty(rows, C, device=DEV, dtype=torch.bfloat16)
    ops.layernorm(x, gamma, beta, 1e-5, out)
    ref = F.layer_norm(x, (C,), gamma, beta, 1e-5)
    assert _rel(out, ref) < 3e-3


# ------------------------------------------------------------------------------------------------ misc
def test_conv_in_out():
    from adaprompt_b200 import ops
    B, H, W = 2, 64, 64
    x = _rand(B, 4, H, W, seed=1)
    w = _rand(320, 4, 3, 3, seed=2, scale=1 / 6.0)
    b = _rand(320, seed=3, scale=0.1)
    y = torch.empty(B, H, W, 320, device=DEV)
    ops.conv_in(x, w, b, y)
    ref = F.conv2d(x, w, b, padding=1).permute(0, 2, 3, 1)
    assert _rel(y, ref) < 1e-5

    xo = _rand(B, H, W, 320, seed=4, dtype=torch.bfloat16)
    wo = _rand(4, 320, 3, 3, seed=5, scale=(9 * 320) ** -0.5)
    bo = _rand(4, seed=6, scale=0.1)
    yo = torch.empty(B, 4, H, W, device=DEV)
    ops.conv_out(xo, wo.permute(0, 2, 3, 1).contiguous(), bo, yo)
    refo = F.conv2d(xo.float().permute(0, 3, 1, 2), wo, bo, padding=1)
    assert _rel(yo, refo) < 1e-5


def test_time_embedding_and_small_linear():
    from adaprompt_b200 import ops
    t = torch.tensor([981.0, 501.0, 21.0, 1.0], device=DEV)
    emb = ops.timestep_embedding(t, 320)
    half = 160
    freqs = torch.exp(-math.log(10000) * torch.arange(half, dtype=torch.float32) / half).to(DEV)
    args = t[:, None] * freqs[None]
    ref = torch.cat([torch.cos(args), torch.sin(args)], -1)
    assert (emb - ref).abs().max().item() < 2e-4

    x = _rand(5, 1280, seed=1)
    w = _rand(640, 1280, seed=2, scale=1280 ** -0.5)
    b = _rand(640, seed=3)
    y = torch.empty(5, 640, device=DEV)
    ops.linear_small(x, w, b, y, silu_in=True, silu_out=True)
    ref = F.silu(F.silu(x) @ w.t() + b)
    assert _rel(y, ref) < 1e-5


def test_casts_and_upsample():
    from adaprompt_b200 import ops
    x = _rand(2, 8, 8, 64, seed=1)
    assert torch.equal(ops.cast_bf16(x), x.to(torch.bfloat16))
    up = torch.empty(2, 16, 16, 64, device=DEV, dtype=torch.bfloat16)
    ops.upsample2x_cast(x, up)
    ref = F.interpolate(x.permute(0, 3, 1, 2), scale_factor=2, mode="nearest").permute(0, 2, 3, 1).to(torch.bfloat16)
    assert torch.equal(up, ref)


def test_cfg_ddim_update_bit_exact():
    """ddim.py:260,279,283,295 in the reference's fp32 operation order -> bit-exact vs torch."""
    from adaprompt_b200 import ops
    b = 3
    x = _rand(b, 4, 64, 64, seed=1)
    eps = _rand(2 * b, 4, 64, 64, seed=2)
    a_t, a_prev, g = torch.tensor(0.3217), torch.tensor(0.3561), 3.6938775510204083
    s1m = torch.sqrt(1 - a_t)
    coef = torch.tensor([[g, s1m.item(), a_t.sqrt().item(), a_prev.sqrt().item(), (1. - a_prev - 0.0).sqrt().item(),
                          0.0, 0, 0]], dtype=torch.float32, device=DEV)
    xp = torch.empty_like(x)
    p0 = torch.empty_like(x)
    ops.cfg_ddim_update(x, eps, coef, xp, p0, has_uncond=True)
    xc, ec = x.cpu(), eps.cpu()
    e_t, e_u = ec.chunk(2)
    e = e_u + g * (e_t - e_u)
    a_t_f = torch.full((b, 1, 1, 1), a_t.item())
    a_prev_f = torch.full((b, 1, 1, 1), a_prev.item())
    sig = torch.full((b, 1, 1, 1), 0.0)
    s1m_f = torch.full((b, 1, 1, 1), s1m.item())
    pred = (xc - s1m_f * e) / a_t_f.sqrt()
    dir_xt = (1. - a_prev_f - sig ** 2).sqrt() * e
    ref = a_prev_f.sqrt() * pred + dir_xt + sig * torch.zeros_like(xc)
    assert torch.equal(p0.cpu(), pred)
    assert torch.equal(xp.cpu(), ref)


def test_cfg_ddim_update_stochastic_bit_exact_in_place():
    """eta > 0, temperature != 1: noise term (sigma * noise) * temperature in the reference's order (ddim.py:286-295);
    the graph path's in-place form (x_prev aliases x) gives the same bits."""
    from adaprompt_b200 import ops
    b = 2
    x = _rand(b, 4, 32, 32, seed=4)
    eps = _rand(2 * b, 4, 32, 32, seed=5)
    noise = _rand(b, 4, 32, 32, seed=6)
    a_t, a_prev, g, sigma, temp = torch.tensor(0.4123), torch.tensor(0.4788), 2.25, torch.tensor(0.1371), 0.85
    s1m = torch.sqrt(1 - a_t)
    coef = torch.tensor([[g, s1m.item(), a_t.sqrt().item(), a_prev.sqrt().item(), (1. - a_prev - sigma ** 2).sqrt().item(),
                          sigma.item(), temp, 0]], dtype=torch.float32, device=DEV)
    xp, p0 = torch.empty_like(x), torch.empty_like(x)
    ops.cfg_ddim_update(x, eps, coef, xp, p0, has_uncond=True, noise=noise)
    xc, ec, nc = x.cpu(), eps.cpu(), noise.cpu()
    e_t, e_u = ec.chunk(2)
    e = e_u + g * (e_t - e_u)
    full = lambda v: torch.full((b, 1, 1, 1), float(v))
    pred = (xc - full(s1m) * e) / full(a_t).sqrt()
    dir_xt = (1. - full(a_prev) - full(sigma) ** 2).sqrt() * e
    ref = full(a_prev).sqrt() * pred + dir_xt + full(sigma) * nc * temp
    assert torch.equal(p0.cpu(), pred)
    assert torch.equal(xp.cpu(), ref)
    x2 = x.clone()
    ops.cfg_ddim_update(x2, eps, coef, x2, p0, has_uncond=True, noise=noise)
    assert torch.equal(x2, xp)


# ------------------------------------------------------------------------------------------------ fused GN statistics
def _group_stats_ref(x, eps):
    """x fp32 [B, HW, C] -> (mean, rstd) [B, 32] in float64."""
    B, HW, C = x.shape
    g = x.double().reshape(B, HW, 32, C // 32)
    mean = g.mean(dim=(1, 3))
    var = g.var(dim=(1, 3), unbiased=False)
    return mean, (var + eps).rsqrt()


@pytest.mark.parametrize("B,HW,N,K,res", [(2, 4096, 320, 320, True), (3, 256, 1280, 640, False), (2, 64, 1280, 1280, True),
                                           (1, 1024, 640, 2560, True)])
def test_gemm_epilogue_gn_stats(B, HW, N, K, res):
    """Statistics written by the GEMM epilogue == statistics of the tensor it wrote; GroupNorm from them."""
    from adaprompt_b200 import ops
    M = B * HW
    a = _rand(M, K, seed=1, dtype=torch.bfloat16)
    w = _rand(N, K, seed=2, scale=K ** -0.5, dtype=torch.bfloat16)
    bias = _rand(N, seed=3)
    r = _rand(M, N, seed=4) if res else None
    out = torch.empty(M, N, device=DEV, dtype=torch.float32)
    st = ops.gn_stats_for_gemm(B, HW, N, DEV)
    assert st is not None
    ops.gemm(a, w, out, bias=bias, residual=r, gn_stats=st.buf)
    part = st.buf.reshape(-1, N, 2)[: M // 32].double()
    rows = out.double().reshape(M // 32, 32, N)
    assert torch.allclose(part[..., 0], rows.sum(1), rtol=1e-5, atol=1e-3)
    assert torch.allclose(part[..., 1], (rows * rows).sum(1), rtol=1e-5, atol=1e-3)
    gamma = 1 + 0.1 * _rand(N, seed=5)
    beta = 0.1 * _rand(N, seed=6)
    y = torch.empty(B, HW, N, device=DEV, dtype=torch.bfloat16)
    ops.groupnorm_apply(out.reshape(B, HW, N), st, gamma, beta, 1e-5, True, y)
    ref = F.silu(F.group_norm(out.reshape(B, HW, N).permute(0, 2, 1), 32, gamma, beta, 1e-5).permute(0, 2, 1))
    assert _rel(y, ref) < 3e-3
    # bit-reproducible
    st2 = ops.gn_stats_for_gemm(B, HW, N, DEV)
    out2 = torch.empty_like(out)
    ops.gemm(a, w, out2, bias=bias, residual=r, gn_stats=st2.buf)
    assert torch.equal(st.buf[: (M // 32) * N * 2], st2.buf[: (M // 32) * N * 2])


@pytest.mark.parametrize("B,H,W,Cin,Cout,stride", [(2, 64, 64, 320, 320, 1), (3, 8, 8, 1280, 1280, 1), (2, 32, 32, 640, 640, 2),
                                                    (1, 24, 24, 640, 320, 1), (2, 16, 16, 1280, 640, 1)])
def test_conv_epilogue_gn_stats_feed_groupnorm(B, H, W, Cin, Cout, stride):
    from adaprompt_b200 import ops
    from adaprompt_b200.packing import pack_conv3x3
    x = _rand(B, H, W, Cin, seed=1, dtype=torch.bfloat16)
    w = _rand(Cout, Cin, 3, 3, seed=2, scale=(9 * Cin) ** -0.5).to(torch.bfloat16)
    bias = _rand(Cout, seed=3)
    Ho, Wo = H // stride, W // stride
    out = torch.empty(B, Ho, Wo, Cout, device=DEV, dtype=torch.float32)
    st = ops.gn_stats_for_conv(B, Ho, Wo, Cout, DEV)
    assert st is not None
    ops.conv3x3(x, pack_conv3x3(w), out, stride=stride, bias=bias, gn_stats=st.buf)
    tot = st.buf.reshape(B, st.slots, Cout, 2).double().sum(1)
    flat = out.double().reshape(B, Ho * Wo, Cout)
    assert torch.allclose(tot[..., 0], flat.sum(1), rtol=1e-5, atol=1e-3)
    assert torch.allclose(tot[..., 1], (flat * flat).sum(1), rtol=1e-5, atol=1e-3)
    # two-source GroupNorm: conv-produced statistics for x0, stand-alone statistics pass for x1
    x1 = _rand(B, Ho, Wo, 320, seed=7) - 0.5
    C = Cout + 320
    gamma = 1 + 0.1 * _rand(C, seed=5)
    beta = 0.1 * _rand(C, seed=6)
    y = torch.empty(B, Ho * Wo, C, device=DEV, dtype=torch.bfloat16)
    raw = torch.empty_like(y)
    ops.groupnorm_apply(out, st, gamma, beta, 1e-6, False, y, x1=x1, st1=ops.groupnorm_stats(x1), raw=raw)
    cat = torch.cat([out, x1], -1).reshape(B, Ho * Wo, C)
    ref = F.group_norm(cat.permute(0, 2, 1), 32, gamma, beta, 1e-6).permute(0, 2, 1)
    assert _rel(y, ref) < 3e-3
    assert torch.equal(raw, cat.to(torch.bfloat16))


def test_conv_gn_slots_small_images_unsupported():
    from adaprompt_b200 import ops
    assert ops.gn_stats_for_conv(2, 4, 4, 1280, DEV) is None      # 16 pixels per sample < one 32-row slot
    assert ops.gn_stats_for_gemm(2, 16, 1280, DEV) is None
    assert ops.gn_stats_for_conv(2, 8, 8, 1280, DEV).slots == 2


def test_conv_out_tensor_core_path():
    """UNetModel.out[-1] (320 -> 4) as an implicit GEMM with Cout padded to 8 + NHWC->NCHW."""
    from adaprompt_b200 import ops
    from adaprompt_b200.unet import UNetModel
    B, H, W, C = 2, 64, 64, 320
    x = _rand(B, H, W, C, seed=1, dtype=torch.bfloat16)
    w = _rand(4, C, 3, 3, seed=2, scale=(9 * C) ** -0.5).to(torch.bfloat16)
    bias = _rand(4, seed=3)
    o8 = torch.empty(B, H, W, 8, device=DEV, dtype=torch.float32)
    ops.conv3x3(x, UNetModel._pad_out_conv(w.float()), o8, bias=UNetModel._pad_out_bias(bias), bn=64)
    out = torch.empty(B, 4, H, W, device=DEV, dtype=torch.float32)
    ops.nhwc_to_nchw(o8, out)
    ref = F.conv2d(x.float().permute(0, 3, 1, 2), w.float(), bias, padding=1)
    assert _rel(out, ref) < 2e-5
    assert o8[..., 4:].abs().max().item() == 0.0


def test_linear_small_many_rows_and_tail_features():
    from adaprompt_b200 import ops
    for M, N, K in [(16, 1280, 320), (33, 1286, 1280), (2, 20480, 1280)]:
        x = _rand(M, K, seed=1)
        w = _rand(N, K, seed=2, scale=K ** -0.5)
        b = _rand(N, seed=3)
        y = torch.empty(M, N, device=DEV)
        ops.linear_small(x, w, b, y, silu_in=True, silu_out=True)
        ref = F.silu(F.silu(x).double() @ w.double().t() + b.double()).float()
        assert _rel(y, ref) < 1e-5


# ------------------------------------------------------------------------------------------------ CTA pairs
@pytest.mark.parametrize("M,N,K,res,bf16out", [(4096, 320, 320, True, False), (1000, 640, 2560, False, True),
                                                (384, 1280, 768, True, True), (65536, 320, 320, True, False)])
def test_gemm_pair_mode_matches_single_cta(M, N, K, res, bf16out):
    """cta_group::2 (two SMs per 256-row tile) and single-CTA schedules accumulate in the same order: bit-identical."""
    from adaprompt_b200 import _lib, ops
    lib = _lib.load()
    a = _rand(M, K, seed=1, dtype=torch.bfloat16)
    w = _rand(N, K, seed=2, scale=K ** -0.5, dtype=torch.bfloat16)
    bias = _rand(N, seed=3)
    r = _rand(M, N, seed=4) if res else None
    outs = []
    for mode in (2, 1):          # AF_PAIR_ALWAYS, AF_PAIR_NEVER (per-call option af_epilogue.pair_mode)
        with ops.launch_options(pair_mode=mode, split_k=1):     # whole tiles: a split tile re-associates the K sum
            out = torch.empty(M, N, device=DEV, dtype=torch.bfloat16 if bf16out else torch.float32)
            ops.gemm(a, w, out, bias=bias, residual=r)
            outs.append(out)
    assert torch.equal(outs[0], outs[1])
    ref = a.float() @ w.float().t() + bias + (r if res else 0)
    assert _rel(outs[0], ref) < (4e-3 if bf16out else 2e-5)


def test_conv_and_geglu_pair_mode_match_single_cta():
    from adaprompt_b200 import _lib, ops
    from adaprompt_b200.packing import pack_conv3x3, pack_geglu
    lib = _lib.load()
    x = _rand(3, 24, 24, 640, seed=1, dtype=torch.bfloat16)
    w = pack_conv3x3(_rand(320, 640, 3, 3, seed=2, scale=(9 * 640) ** -0.5).to(torch.bfloat16))
    res = _rand(3, 24, 24, 320, seed=5)
    a = _rand(2048, 320, seed=3, dtype=torch.bfloat16)
    wg, bg = pack_geglu(_rand(2560, 320, seed=4, scale=320 ** -0.5), _rand(2560, seed=6))
    wg = wg.to(torch.bfloat16).contiguous()
    outs = []
    for mode in (2, 1):
        with ops.launch_options(pair_mode=mode, split_k=1):
            o1 = torch.empty(3, 24, 24, 320, device=DEV)
            st = ops.gn_stats_for_conv(3, 24, 24, 320, DEV)
            ops.conv3x3(x, w, o1, residual=res, gn_stats=st.buf)
            o2 = torch.empty(2048, 1280, device=DEV, dtype=torch.bfloat16)
            ops.gemm(a, wg, o2, bias=bg, geglu=True)
            outs.append((o1, st.buf.clone(), o2))
    for u, v in zip(*outs):
        assert torch.equal(u, v)


# ------------------------------------------------------------------------------------------------ split-K of the last wave
def _splitk_flags_clear():
    from adaprompt_b200 import ops
    torch.cuda.synchronize()
    return all(int(st[k][:4096].view(torch.int32).abs().sum().item()) == 0
               for st in ops._splitk_ws.values() for k in ("eager", "graph"))


@pytest.mark.parametrize("M,N,K,bn,res,bf16out,split", [
    (1024, 1280, 1280, 0, True, False, 0),      # 64 tiles on 148 SMs: the auto plan splits
    (1024, 1280, 2560, 0, False, False, 5),
    (4096, 1280, 1280, 0, True, False, 0),      # 256 tiles = one full wave + 108 remainder tiles
    (4096, 1280, 5120, 0, True, True, 4),
    (1000, 640, 2560, 128, False, True, 3),     # ragged M, last K range shorter than the others
    (300, 320, 320, 0, True, False, 2),
])
def test_gemm_split_k_matches_whole_tiles(M, N, K, bn, res, bf16out, split):
    """The K ranges of a split tile are summed in range order: deterministic, equal to the whole-tile schedule up to
    fp32 re-association (1e-6), flags left clear for the next launch."""
    from adaprompt_b200 import ops
    a = _rand(M, K, seed=1, dtype=torch.bfloat16)
    w = _rand(N, K, seed=2, scale=K ** -0.5, dtype=torch.bfloat16)
    bias = _rand(N, seed=3)
    r = _rand(M, N, seed=4) if res else None
    dt = torch.bfloat16 if bf16out else torch.float32
    outs = {}
    for mode in (1, split, split):
        with ops.launch_options(split_k=mode):
            out = torch.empty(M, N, device=DEV, dtype=dt)
            st = ops.gn_stats_for_gemm(1, ((M + 31) // 32) * 32, N, DEV) if (not bf16out and M % 32 == 0) else None
            ops.gemm(a, w, out, bias=bias, residual=r, bn=bn, gn_stats=st.buf if st else None)
            outs.setdefault(mode, []).append((out, st.buf.clone() if st else None))
    whole, (s1, s2) = outs[1][0], outs[split]
    assert torch.equal(s1[0], s2[0]) and (s1[1] is None or torch.equal(s1[1], s2[1]))        # run-to-run bit-exact
    ref = a.float() @ w.float().t() + bias + (r if res else 0)
    assert _rel(s1[0], ref) < (4e-3 if bf16out else 2e-5)
    assert _rel(s1[0], whole[0]) < (4e-3 if bf16out else 1e-5)
    if s1[1] is not None:
        assert _rel(s1[1], whole[1]) < 1e-5
    assert _splitk_flags_clear()


@pytest.mark.parametrize("B,H,W,C0,C1,Cout,stride,split", [
    (16, 8, 8, 1280, 0, 1280, 1, 0), (16, 8, 8, 1280, 1280, 1280, 1, 9), (16, 16, 16, 1280, 0, 1280, 2, 0),
    (4, 8, 8, 1280, 0, 1280, 1, 0), (2, 16, 16, 640, 320, 640, 1, 7), (16, 16, 16, 1280, 0, 1280, 1, 0),
])
def test_conv_split_k_matches_whole_tiles(B, H, W, C0, C1, Cout, stride, split):
    from adaprompt_b200 import ops
    from adaprompt_b200.packing import pack_conv3x3
    Cin = C0 + C1
    x0 = _rand(B, H, W, C0, seed=1, dtype=torch.bfloat16)
    x1 = _rand(B, H, W, C1, seed=2, dtype=torch.bfloat16) if C1 else None
    wt = _rand(Cout, Cin, 3, 3, seed=3, scale=(9 * Cin) ** -0.5).to(torch.bfloat16)
    w = pack_conv3x3(wt)
    bias, emb = _rand(Cout, seed=4), _rand(B, Cout, seed=5)
    Ho, Wo = H // stride, W // stride
    res = _rand(B, Ho, Wo, Cout, seed=6)
    outs = []
    for mode in (1, split):
        with ops.launch_options(split_k=mode):
            out = torch.empty(B, Ho, Wo, Cout, device=DEV)
            st = ops.gn_stats_for_conv(B, Ho, Wo, Cout, DEV)
            ops.conv3x3(x0, w, out, x1=x1, stride=stride, bias=bias, rowbias=emb, residual=res,
                        gn_stats=st.buf if st else None)
            outs.append((out, st.buf.clone() if st else None))
    ref = _conv_ref(torch.cat([x0, x1], -1) if C1 else x0, wt, bias, stride) + emb[:, None, None, :] + res
    assert _rel(outs[1][0], ref) < 2e-5
    assert _rel(outs[1][0], outs[0][0]) < 5e-5          # fp32 re-association of the K = 9 * Cin sum
    if outs[0][1] is not None:
        assert _rel(outs[1][1], outs[0][1]) < 1e-5
    assert _splitk_flags_clear()


def test_split_k_replays_from_a_cuda_graph():
    from adaprompt_b200 import ops
    from adaprompt_b200.packing import pack_conv3x3
    x = _rand(16, 8, 8, 1280, seed=1, dtype=torch.bfloat16)
    w = pack_conv3x3(_rand(1280, 1280, 3, 3, seed=2, scale=(9 * 1280) ** -0.5).to(torch.bfloat16))
    out = torch.empty(16, 8, 8, 1280, device=DEV)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    ops.conv3x3(x, w, out)                     # an eager launch creates the workspaces outside the capture
    eager = out.clone()
    torch.cuda._sleep(400_000_000)             # keeps the first stream busy for ~0.2 s
    with torch.cuda.stream(side):              # a second eager stream gets the whole-tile schedule while the first has
        assert ops._splitk_workspace(out.device) is None              # work in flight (see ops._splitk_workspace)
        side_out = torch.empty_like(out)
        ops.conv3x3(x, w, side_out)
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        ops.conv3x3(x, w, out)
        ops.conv3x3(x, w, out)
    for _ in range(3):
        out.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, eager)
    assert _splitk_flags_clear()
    with ops.launch_options(split_k=1):
        whole = torch.empty_like(out)
        ops.conv3x3(x, w, whole)
    assert not torch.equal(whole, eager) and _rel(whole, eager) < 5e-5     # the captured launches did split
    assert torch.equal(side_out, whole)
