"""The Stage-1 step on image-masked batches on a B200: the key-masked attention backward (fused tcgen05 kernels and the
masked bgemm modes) against a float64 restatement of the masked_fill softmax of attention.py:223-232, the masked context
gradient of the UNet against autograd through the CPU oracle, and the masked DistillStep / Stage1Trainer paths."""
import math

import pytest
import torch
import torch.nn.functional as F

from test_train_gpu import (COMPOSED_TOL, DEV, FUSED_TOL, LN2, _attn_bwd_inputs, _check_grads, _clip_small, _kernels,
                            _rel, _rows_bf16, _sbg_small, _unet)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False


# ------------------------------------------------------------------------------------------------ reference
def _masked_ref(qs, k, v, dO, m):
    """Masked attention forward / backward in float64 (qs, k, v, dO [B, n, h, d], m bool [B, nk]), per sample:
    a sample with a kept key: softmax over its kept keys, masked P and dS exactly 0; a sample that keeps none: P = 1/nk,
    dS = 0 (masked_fill passes no gradient), lse = +inf.  Returns O, dQ, dK, dV [B, n, h, d], lse, delta [B, h, Nq]."""
    B, Nq, h, d = qs.shape
    nk = k.shape[1]
    f64 = dict(dtype=torch.float64, device=qs.device)
    r = {"O": torch.empty(B, Nq, h, d, **f64), "dQ": torch.empty(B, Nq, h, d, **f64),
         "dK": torch.empty(B, nk, h, d, **f64), "dV": torch.empty(B, nk, h, d, **f64),
         "lse": torch.empty(B, h, Nq, **f64), "delta": torch.empty(B, h, Nq, **f64)}
    for b in range(B):
        keep = m[b].to(qs.device)
        for j in range(h):
            q_, k_, v_, g_ = (t[b, :, j].double() for t in (qs, k, v, dO))
            s = (q_ @ k_.t()) * LN2
            if keep.any():
                s = s.masked_fill(~keep[None], -math.inf)
                lse = torch.logsumexp(s, -1)
                p = torch.exp(s - lse[:, None])
                lse = lse / LN2
            else:
                p = torch.full_like(s, 1.0 / nk)
                lse = torch.full((Nq,), math.inf, **f64)
            del s
            o = p @ v_
            delta = (g_ * o).sum(-1)
            ds = p * (g_ @ v_.t() - delta[:, None]) if keep.any() else torch.zeros_like(p)
            r["O"][b, :, j], r["lse"][b, j], r["delta"][b, j] = o, lse, delta
            r["dV"][b, :, j] = p.t() @ g_
            r["dQ"][b, :, j] = LN2 * (ds @ k_)
            r["dK"][b, :, j] = LN2 * (ds.t() @ q_)
    return r


def test_masked_reference_matches_masked_fill_autograd():
    """_masked_ref against torch.autograd through masked_fill(-finfo.max) + softmax (oracle/unet_oracle.py:233-236), in
    float64, with a sample that keeps no key."""
    B, N, h, d = 3, 24, 2, 8
    g = torch.Generator().manual_seed(1)
    qs, k, v, dO = (torch.randn(B, N, h, d, generator=g, dtype=torch.float64) for _ in range(4))
    m = torch.rand(B, N, generator=g) < 0.5
    m[0] = False
    m[1, 3] = True
    ref = _masked_ref(qs, k, v, dO, m)
    qa, ka, va = (t.clone().requires_grad_(True) for t in (qs, k, v))
    s = torch.einsum("bihd,bjhd->bhij", qa, ka) * LN2
    s = s.masked_fill(~m[:, None, None, :], -torch.finfo(torch.float64).max)
    o = torch.einsum("bhij,bjhd->bihd", torch.softmax(s, -1), va)
    o.backward(dO)
    for name, want in (("O", o), ("dQ", qa.grad), ("dK", ka.grad), ("dV", va.grad)):
        assert torch.allclose(ref[name], want.detach(), rtol=1e-10, atol=1e-12), name


def _grid(N):
    w = max(x for x in range(1, int(math.isqrt(N)) + 1) if N % x == 0)
    return N // w, w


def _mask(regime, B, N, seed):
    """bool [B, N] key masks:
      random: 50 % kept;  one: one kept key;  rect: a face-like rectangle of the H x W token grid;
      last: one kept key, in the last 64-key block;  mixed: sample 0 keeps no key, the others random;
      poison: random (the caller fills the masked K / V rows with large values)."""
    g = torch.Generator().manual_seed(seed)
    m = torch.rand(B, N, generator=g) < 0.5
    if regime == "one":
        m = torch.zeros(B, N, dtype=torch.bool)
        m[torch.arange(B), torch.randint(0, N, (B,), generator=g)] = True
    elif regime == "rect":
        H, W = _grid(N)
        m = torch.zeros(B, H, W, dtype=torch.bool)
        for b in range(B):
            m[b, H // 4 + b % 2:H - H // 5, W // 6:W - W // 3 + b % 2] = True
        m = m.reshape(B, N)
    elif regime == "last":
        m = torch.zeros(B, N, dtype=torch.bool)
        lo = (N - 1) // 64 * 64
        m[torch.arange(B), lo + torch.randint(0, N - lo, (B,), generator=g)] = True
    elif regime == "mixed":
        m[0] = False
    m[m.sum(1) == 0 if regime != "mixed" else torch.zeros(B, dtype=torch.bool), 0] = True
    return m


def _poison(kb, vb, m, B, n, seed=99):
    """Masked K rows scaled by 2^10, masked V rows +-2^100 (bf16 [B*n, cols] buffers, in place)."""
    gen = torch.Generator().manual_seed(seed)
    drop = (~m).to(DEV).reshape(B * n, 1)
    kb.copy_(torch.where(drop, (kb.float() * 1024).to(kb.dtype), kb))
    sign = (torch.randint(0, 2, vb.shape, generator=gen) * 2 - 1).to(DEV)
    vb.copy_(torch.where(drop, (sign * 2.0 ** 100).to(vb.dtype), vb))


def _zero_masked_rows(t, m):
    """[B, n, h, d] with the rows of masked keys zeroed: the run every other content of those rows must reproduce."""
    return t * m.to(t.device)[:, :, None, None]


# Regimes in which every sample keeps exactly one key: softmax rows are one-hot, dS = P o (dP - delta) is 0 exactly, so
# dQ and dK are 0 up to rounding (what remains of T - delta in fp32): checked by their largest entry, not relatively.
# Largest |dQ|, |dK| seen on one B200 (1000 W): 1.2e-5 (fused), 3.0e-5 (bgemm path); limit 6e-5.
ONE_KEY = ("one", "last")
ONE_KEY_ABS = 6e-5


def _check_one_key(label, got, ref, tol):
    from test_train_gpu import _grad_errors
    big = {g: got[g].abs().max().item() for g in ("dQ", "dK")}
    e = _grad_errors(got["dV"], ref["dV"])
    print(f"\n{label}: one kept key per sample, largest |dQ| {big['dQ']:.2e} |dK| {big['dK']:.2e}, dV rel {e['rel']:.2e} "
          f"row {e['row']:.2e}")
    assert big["dQ"] < ONE_KEY_ABS and big["dK"] < ONE_KEY_ABS, (label, big)
    assert e["rel"] < tol["dV"][0] and e["row"] < tol["dV"][1], (label, e)


def _check_masked_zeros(label, dq, dk, dv, m):
    """Exact zeros: dK / dV rows of masked keys in samples that keep a key; dQ and dK of samples that keep none."""
    m = m.to(dq.device)
    empty = m.sum(1) == 0
    drop = ~m & ~empty[:, None]
    assert not dk[drop].any() and not dv[drop].any(), f"{label}: dK / dV rows of masked keys"
    assert not dq[empty].any() and not dk[empty].any(), f"{label}: dQ / dK of a sample that keeps no key"


# ------------------------------------------------------------------------------------------------ fused kernels
REGIMES = ("random", "one", "rect", "last", "mixed", "poison")
FUSED_MASK_CASES = (
    [pytest.param(B, N, d, r, id=f"d{d}-B{B}-N{N}-{r}") for d, B, N in ((40, 4, 128), (40, 2, 1024), (80, 4, 256),
                                                                         (80, 2, 1024)) for r in REGIMES]
    + [pytest.param(B, N, d, r, id=f"d{d}-B{B}-N{N}-{r}") for d, B, N in ((40, 2, 4096), (80, 2, 2304), (40, 2, 9216))
       for r in ("rect", "mixed")]
    + [pytest.param(8, 1024, 40, "random", id="d40-B8-N1024-random")])


def _fused_operands(qs, k, v, g, dp):
    q, kk, vp, dop = _rows_bf16(qs, dp), _rows_bf16(k, dp), _rows_bf16(v, dp), _rows_bf16(g, dp)
    return q, kk, vp, dop


def _fused_call(q, kk, vp, dop, ref, B, N, d, heads, km):
    from adaprompt_b200 import ops
    qT, kT, dOT = (t.t().contiguous() for t in (q, kk, dop))
    return ops.attention_bwd(q, kk, vp, dop, qT, kT, dOT, ref["lse"].float(), ref["delta"].float(), B=B, heads=heads,
                             N=N, d=d, key_mask=km)


@pytest.mark.parametrize("B,N,d,regime", FUSED_MASK_CASES)
def test_attention_bwd_masked_fused_kernel(B, N, d, regime):
    """ops.attention_bwd with a key mask, lse and delta from the float64 reference, the masked K / V rows holding random
    values (the masked_fill reference ignores them; dQ_i = ln2 sum_j dS_ij K_j, so a masked dS column the kernel failed
    to zero would reach dQ): FUSED_TOL, exact zeros where the mask owes them, and the unmasked kernels on the same
    operands shown to miss FUSED_TOL by far (the test sees a dropped mask).  The gradients are bit-identical to those
    with zeros in the masked rows, and in the poison regime also with those rows' K scaled by 2^10 and V = +-2^100."""
    from test_train_gpu import _grad_errors
    from adaprompt_b200.packing import head_pad
    heads, dp = 8, head_pad(d)
    qs, k, v, g = _attn_bwd_inputs(B, N, N, heads, d, seed=N + d + B)
    m = _mask(regime, B, N, seed=N + B)
    km = m.to(torch.uint8).to(DEV)
    ref = _masked_ref(qs, k, v, g, m)
    q, kk, vp, dop = _fused_operands(qs, k, v, g, dp)
    raw = dq, dk, dv = _fused_call(q, kk, vp, dop, ref, B, N, d, heads, km)
    for t in (dq, dk, dv):
        assert torch.isfinite(t.float()).all()
    dq, dk, dv = dq.view(B, N, heads, dp), dk.view(B, N, heads, dp), dv.view(B, N, heads, d)
    assert not dq[..., d:].any() and not dk[..., d:].any(), "pad columns of dQ / dK"
    label = f"masked fused B={B} N={N} d={d} {regime} (kept {int(m.sum())}/{B * N})"
    _check_masked_zeros(label, dq, dk, dv, m)
    got = {"dQ": dq[..., :d], "dK": dk[..., :d], "dV": dv}
    if regime in ONE_KEY:
        _check_one_key(label, got, ref, FUSED_TOL)
    else:
        _check_grads(label, got, ref, FUSED_TOL)
    # the same operands through the unmasked kernels: dQ far outside the limits
    uq = _fused_call(q, kk, vp, dop, ref, B, N, d, heads, None)[0].view(B, N, heads, dp)[..., :d]
    if regime in ONE_KEY:
        miss = uq.abs().max().item()
        print(f"{label}: unmasked kernels, largest |dQ| {miss:.2e}")
        assert miss > 100 * ONE_KEY_ABS, (label, miss)
    else:
        miss = _grad_errors(uq, ref["dQ"])["rel"]
        print(f"{label}: unmasked kernels, dQ rel {miss:.2e}")
        assert miss > 5 * FUSED_TOL["dQ"][0], (label, miss)
    # masked rows: zeros, and (poison) 2^10 K / +-2^100 V, against the random rows above, bit for bit
    variants = [_fused_operands(qs, _zero_masked_rows(k, m), _zero_masked_rows(v, m), g, dp)]
    if regime == "poison":
        kp, vpp = kk.clone(), vp.clone()
        _poison(kp, vpp, m, B, N)
        variants.append((q, kp, vpp, dop))
    for ops_ in variants:
        other = _fused_call(*ops_, ref, B, N, d, heads, km)
        for a, b_ in zip(raw, other):
            assert torch.equal(a.reshape(-1).view(torch.int16), b_.reshape(-1).view(torch.int16)), label


@pytest.mark.parametrize("B,N,d", [(2, 128, 40), (2, 1024, 40), (2, 256, 80), (1, 2304, 80)])
def test_attention_bwd_masked_all_ones_is_bit_identical(B, N, d):
    from adaprompt_b200 import ops
    from adaprompt_b200.packing import head_pad
    heads, dp = 8, head_pad(d)
    qs, k, v, g = _attn_bwd_inputs(B, N, N, heads, d, seed=7)
    ref = _masked_ref(qs, k, v, g, torch.ones(B, N, dtype=torch.bool))
    q, kk, vp, dop = _fused_operands(qs, k, v, g, dp)
    qT, kT, dOT = (t.t().contiguous() for t in (q, kk, dop))
    plain = ops.attention_bwd(q, kk, vp, dop, qT, kT, dOT, ref["lse"].float(), ref["delta"].float(), B=B, heads=heads,
                              N=N, d=d)
    masked = _fused_call(q, kk, vp, dop, ref, B, N, d, heads, torch.ones(B, N, dtype=torch.uint8, device=DEV))
    for a, b_ in zip(plain, masked):
        assert torch.equal(a.view(torch.int16), b_.view(torch.int16))


# ------------------------------------------------------------------------------------------------ AttentionFn
def _attention_fn_masked(qs, k, v, g, m, fused, poison=False):
    """AttentionFn forward + backward with key_mask on the UNet's [Q|K] self-attention layout.  fused = False sets
    ops.attention_bwd to None (the bgemm path).  -> o, dq [B*N, h*dp], dk, dv."""
    from adaprompt_b200 import ops
    from adaprompt_b200.packing import head_pad
    from adaprompt_b200.train import AttentionFn
    B, N, h, d = qs.shape
    dp = head_pad(d)
    kb, vb = _rows_bf16(k, dp), _rows_bf16(v, d)
    if poison:
        _poison(kb, vb, m, B, N)
    qk = torch.cat([_rows_bf16(qs, dp), kb], 1)
    q, kk = qk.detach().requires_grad_(True), qk[:, h * dp:].detach().requires_grad_(True)
    vv = vb.requires_grad_(True)
    km = m.to(torch.uint8).to(DEV)
    orig = ops.attention_bwd
    if not fused:
        ops.attention_bwd = None
    try:
        o = AttentionFn.apply(q, kk, vv, B, h, d, N, N, N, km)
        o.backward(g.reshape(B * N, h * d).to(torch.bfloat16))
    finally:
        ops.attention_bwd = orig
    return o.detach(), q.grad[:, :h * dp], kk.grad, vv.grad


def _attention_fn_masked_case(B, N, d, regime, fused, seed=3):
    from adaprompt_b200.packing import head_pad
    h, dp = 8, head_pad(d)
    qs, k, v, g = _attn_bwd_inputs(B, N, N, h, d, seed=seed)
    m = _mask(regime, B, N, seed=seed + N)
    ref = _masked_ref(qs, k, v, g, m)          # masked K / V rows keep their random values: the reference ignores them
    o, dq, dk, dv = _attention_fn_masked(qs, k, v, g, m, fused)
    label = f"AttentionFn masked {'fused' if fused else 'bgemm'} B={B} N={N} d={d} {regime}"
    assert _rel(o.view(B, N, h, d), ref["O"]) < 1e-2, label
    dq, dk, dv = dq.reshape(B, N, h, dp), dk.reshape(B, N, h, dp), dv.reshape(B, N, h, d)
    for t in (dq, dk, dv):
        assert torch.isfinite(t.float()).all(), label
    _check_masked_zeros(label, dq, dk, dv, m)
    got = {"dQ": dq[..., :d], "dK": dk[..., :d], "dV": dv}
    if regime in ONE_KEY:
        _check_one_key(label, got, ref, COMPOSED_TOL)
    else:
        _check_grads(label, got, ref, COMPOSED_TOL)
    # masked rows holding zeros, and (poison) 2^10 K / +-2^100 V: the same gradients bit for bit
    runs = [_attention_fn_masked(qs, _zero_masked_rows(k, m), _zero_masked_rows(v, m), g, m, fused)]
    if regime == "poison":
        runs.append(_attention_fn_masked(qs, k, v, g, m, fused, poison=True))
    for _, dq2, dk2, dv2 in runs:
        for a, b_ in zip((dq, dk, dv), (dq2, dk2, dv2)):
            assert torch.equal(a.reshape(-1).view(torch.int16), b_.reshape(-1).view(torch.int16)), label


@pytest.mark.parametrize("regime", REGIMES)
@pytest.mark.parametrize("B,N,d", [(2, 16, 160), (2, 64, 160), (2, 256, 160), (2, 200, 40)])
def test_attention_backward_masked_bgemm_path(B, N, d, regime):
    _attention_fn_masked_case(B, N, d, regime, fused=False)


@pytest.mark.parametrize("B,N,d", [(2, 64, 160), (2, 200, 40), (2, 256, 80)])
def test_masked_bgemm_all_ones_is_bit_identical(B, N, d):
    from adaprompt_b200 import ops
    from adaprompt_b200.packing import head_pad
    from adaprompt_b200.train import AttentionFn
    h, dp = 8, head_pad(d)
    qs, k, v, g = _attn_bwd_inputs(B, N, N, h, d, seed=4)
    grads = []
    for km in (None, torch.ones(B, N, dtype=torch.uint8, device=DEV)):
        qk = torch.cat([_rows_bf16(qs, dp), _rows_bf16(k, dp)], 1)
        q, kk = qk.detach().requires_grad_(True), qk[:, h * dp:].detach().requires_grad_(True)
        vv = _rows_bf16(v, d).requires_grad_(True)
        orig, ops.attention_bwd = ops.attention_bwd, None
        try:
            args = (q, kk, vv, B, h, d, N, N, N) + ((km,) if km is not None else ())
            AttentionFn.apply(*args).backward(g.reshape(B * N, h * d).to(torch.bfloat16))
        finally:
            ops.attention_bwd = orig
        grads.append((q.grad, kk.grad, vv.grad))
    for a, b_ in zip(*grads):
        assert torch.equal(a.view(torch.int16), b_.view(torch.int16))


@pytest.mark.parametrize("B,N,d,regime", [(2, 1024, 40, "rect"), (2, 256, 80, "mixed"), (2, 512, 40, "poison"),
                                          (2, 4096, 40, "mixed")])
def test_attention_fn_masked_fused_end_to_end(B, N, d, regime):
    """AttentionFn with a key mask through the masked forward (lse = +inf rows included) and the fused backward."""
    _attention_fn_masked_case(B, N, d, regime, fused=True)


def test_masked_backward_runs_the_masked_kernels():
    """The profiler sees attention_bwd_masked_kernel (all four instantiations) on fused-eligible shapes and
    bgemm_masked_kernel (modes 1-4) elsewhere; no unmasked softmax-epilogue kernel runs under a mask."""
    seen = set()
    for B, N, d in ((1, 256, 40), (1, 256, 80), (2, 64, 160), (1, 200, 40)):
        qs, k, v, g = _attn_bwd_inputs(B, N, N, 8, d, seed=2)
        m = _mask("random", B, N, 1)
        with _kernels() as names:
            _attention_fn_masked(qs, k, v, g, m, fused=True)
        fused = any("attention_bwd_masked_kernel" in n for n in names)
        assert fused == (d in (40, 80) and N % 128 == 0), (B, N, d, names)
        assert not any("attention_bwd_kernel" in n for n in names)
        assert not any(f"bgemm_kernel<{bn},{mode}>" in n for bn in (64, 128) for mode in (1, 2, 3, 4) for n in names)
        seen.update(names)
    want = [f"attention_bwd_masked_kernel<{d},{dkv}>" for d in (40, 80) for dkv in ("false", "true")]
    want += [f"bgemm_masked_kernel<{bn},{mode}>" for bn in (64, 128) for mode in (1, 2, 3, 4)]
    missing = [w for w in want if not any(w in n for n in seen)]
    assert not missing, (missing, sorted(n for n in seen if "bwd" in n or "bgemm" in n))


# ------------------------------------------------------------------------------------------------ whole UNet
def _unet_masks(B, H, seed):
    g = torch.Generator().manual_seed(seed)
    m = torch.zeros(B, 1, H, H)
    m[0, :, 9:16, 5:27] = 1                    # rectangle between rows 8 and 16: nearest to 4x4 samples rows 0, 8, 16, 24
    m[1] = (torch.rand(1, H, H, generator=g) < 0.6).float()
    return m


def test_unet_context_gradient_with_image_mask_matches_oracle_autograd():
    """d loss / d context with an image mask (batch 2, 32x32 latent; one rectangle, one random mask) against autograd
    through the fp32 CPU oracle, with the masked loss (budgets of test_unet_context_gradient_matches_oracle_autograd).
    An all-ones mask gives the unmasked gradient up to bf16 noise: the masked self-attention FORWARD runs another kernel
    than the unmasked one (its backward is bit-identical, test_attention_bwd_masked_all_ones_is_bit_identical), and
    its roundings travel through the 25 blocks of the backward.  Measured 6.5e-3 on one B200 (1000 W); limit 1.3e-2."""
    from adaprompt_b200.train import calc_recon_loss, distill_loss, unet_forward_train
    from oracle.golden_inputs import EXTRA_INFO
    from oracle.unet_oracle import UNetSpec, unet_forward
    unet, sd = _unet()
    g = torch.Generator().manual_seed(17)
    B, H = 2, 32
    x = torch.randn(B, 4, H, H, generator=g)
    t = torch.tensor([501, 121])
    ctx = torch.randn(16 * B, 77, 768, generator=g)
    target = torch.randn(B, 4, H, H, generator=g)
    mask = _unet_masks(B, H, 3)
    m4 = F.interpolate(mask, size=(4, 4), mode="nearest").reshape(B, -1)
    assert m4[0].sum() == 0 and m4[1].sum() > 0, "the 4x4 level must see a sample that keeps no key"
    c_ref = ctx.clone().requires_grad_(True)
    eps_ref = unet_forward(sd, UNetSpec(), x, t, c_ref, dict(EXTRA_INFO, img_mask=mask))
    loss_ref = calc_recon_loss(eps_ref, target, mask)
    loss_ref.backward()
    c = ctx.to(DEV).requires_grad_(True)
    eps = unet_forward_train(unet, x.to(DEV), t.to(DEV), c, dict(EXTRA_INFO, img_mask=mask.to(DEV)))
    loss = calc_recon_loss(eps, target.to(DEV), mask.to(DEV))
    loss.backward()
    e_eps = _rel(eps, eps_ref)
    err = _rel(c.grad, c_ref.grad)
    per_layer = [_rel(c.grad.reshape(B, 16, 77, 768)[:, l], c_ref.grad.reshape(B, 16, 77, 768)[:, l]) for l in range(16)]
    print(f"\nmasked UNet: eps rel-L2 {e_eps:.2e}, loss {loss.item():.6f} vs {loss_ref.item():.6f}, context grad rel-L2 "
          f"{err:.2e}, per layer max {max(per_layer):.2e}", [f"{e:.3f}" for e in per_layer])
    assert e_eps < 1e-2
    assert abs(loss.item() - loss_ref.item()) < 1e-2 * abs(loss_ref.item())
    assert err < 2e-2 and max(per_layer) < 6e-2, (err, per_layer)
    # all-ones image mask against no mask
    ones = torch.ones(B, 1, H, H, device=DEV)
    grads = []
    for extra in (dict(EXTRA_INFO), dict(EXTRA_INFO, img_mask=ones)):
        c = ctx.to(DEV).requires_grad_(True)
        distill_loss(unet_forward_train(unet, x.to(DEV), t.to(DEV), c, extra), target.to(DEV)).backward()
        grads.append(c.grad)
    e1 = _rel(grads[1], grads[0])
    print(f"all-ones image mask vs none: context grad rel-L2 {e1:.2e}")
    assert e1 < 1.3e-2


# ------------------------------------------------------------------------------------------------ DistillStep / trainer
def _stack():
    from adaprompt_b200.train_cond import DistillStep
    from oracle import text_oracle as to
    from oracle.unet_oracle import make_alphas_cumprod
    from test_text_gpu import StubTokenizer
    unet, sd_unet = _unet()
    sbg, sd_sbg = _sbg_small(31, 2)
    frozen, sd_frozen = _clip_small(32, 2)
    arc2face, sd_arc = _clip_small(33, 2)
    frozen.text_model.last_layers_skip_weights = [0.5, 0.5]
    for m in (frozen, arc2face):
        for p in m.parameters():
            p.requires_grad = False
    acp = torch.tensor(make_alphas_cumprod(), dtype=torch.float32)
    step = DistillStep(unet, frozen.text_model, sbg, arc2face.eval(), StubTokenizer(), acp, to.TOK_Z,
                       fg_pixel_weight=2.0, bg_pixel_weight=0.5)
    return step, sbg, (sd_unet, sd_sbg, sd_frozen, sd_arc), acp


def test_distill_step_with_masks_end_to_end_gradients():
    """Whole masked micro-step (batch 2, 32x32 latent, 2-layer CLIPs, fg / bg pixel weights 2 and 0.5): the
    SubjBasisGenerator gradients against autograd through the conditioning and UNet oracles and calc_recon_loss."""
    from adaprompt_b200.synthetic import synthetic_masks
    from adaprompt_b200.train import calc_recon_loss
    from oracle import text_oracle as to
    from oracle.golden_inputs import EXTRA_INFO
    from oracle.unet_oracle import UNetSpec, unet_forward
    from test_train_gpu import _cond_reference
    step, sbg, (sd_unet, sd_sbg, sd_frozen, sd_arc), acp = _stack()
    g = torch.Generator().manual_seed(9)
    B = 2
    img, fg = synthetic_masks(B, 32, torch.Generator().manual_seed(4))
    batch = {"x0": torch.randn(B, 4, 32, 32, generator=g), "noise": torch.randn(B, 4, 32, 32, generator=g),
             "t": torch.tensor([601, 141]), "teacher_eps": torch.randn(B, 4, 32, 32, generator=g),
             "face_embs": F.normalize(torch.randn(B, 512, generator=g), dim=-1),
             "tokens": torch.tensor([to.subject_prompt_ids(77)] * B), "img_mask": img, "fg_mask": fg}
    sd_ref = {k: v.clone().requires_grad_(True) for k, v in sd_sbg.items()}
    hw_ref = torch.tensor([[1.0], [2.0], [4.0]], requires_grad=True)
    with torch.no_grad():
        _, id_embs = to.arc2face_forward_face_embs(sd_arc, batch["face_embs"])
    c_ref = _cond_reference(sd_ref, sd_frozen, hw_ref, id_embs, batch["tokens"])
    a = acp[batch["t"]].view(-1, 1, 1, 1)
    x_noisy = a.sqrt() * batch["x0"] + (1 - a).sqrt() * batch["noise"]
    eps_ref = unet_forward(sd_unet, UNetSpec(), x_noisy, batch["t"], c_ref, dict(EXTRA_INFO, img_mask=img))
    loss_ref = calc_recon_loss(eps_ref, batch["teacher_eps"], img, fg, 2.0, 0.5)
    loss_ref.backward()
    loss = step.micro_step({k: v.cuda() for k, v in batch.items()})
    scale = sbg.prompt2token_proj_grad_scale
    worst = ("", 0.0)
    for name, p in sbg.prompt2token_proj.named_parameters():
        ref = sd_ref[name].grad
        if name.endswith("token_embedding.weight") or name.endswith("k_proj.bias") or ref is None or ref.abs().max() == 0:
            continue
        worst = max(worst, (name, _rel(p.grad / scale, ref)), key=lambda t: t[1])
    print(f"\nmasked end-to-end: loss {loss:.6f} vs {loss_ref.item():.6f}, worst parameter gradient {worst}")
    assert abs(loss - loss_ref.item()) < 1e-2 * abs(loss_ref.item())
    assert worst[1] < 3e-2, worst


def test_stage1_trainer_with_masks():
    """Stage1Trainer on masked batches: graph and eager buckets agree (1e-5) over two replays with new masks; fused
    micro-batches agree with the loop (5e-3); alternating masked and unmasked steps recapture, and the unmasked steps
    give the loss of a trainer that never saw a mask bit for bit, and its bucket up to the order of the atomic sums in
    the parameter-gradient kernels (token-embedding scatter-add, LayerNorm dgamma / dbeta: two trainers that never see a
    mask differ the same way); mismatched mask sets raise ValueError."""
    from adaprompt_b200.synthetic import stage1_batch
    from adaprompt_b200.train_cond import Stage1Trainer, trainable_parameters
    from oracle import text_oracle as to
    step, sbg, _, _ = _stack()
    params = trainable_parameters(sbg)
    gen = torch.Generator().manual_seed(19)

    def batch(masks):
        b = stage1_batch(DEV, 2, 32, gen, masks=masks)
        b["tokens"] = torch.tensor([to.subject_prompt_ids(77)] * 2, device=DEV)
        return b

    class NoOpt:
        def step(self, flat):
            self.seen = flat.clone()

    eager = Stage1Trainer(step, params, accum=2, use_graph=False, optimizer=NoOpt())
    graph = Stage1Trainer(step, params, accum=2, use_graph=True, optimizer=NoOpt())
    whole = Stage1Trainer(step, params, accum=2, use_graph="step", optimizer=NoOpt())
    whole._gstep.fuse_unet = False
    fused = Stage1Trainer(step, params, accum=2, use_graph="step", optimizer=NoOpt())
    for rep in range(2):
        bs = [batch(True), batch(True)]
        o_e = eager.optimizer_step(bs)
        for tr in (graph, whole):
            o_g = tr.optimizer_step(bs)
            e = _rel(tr.optimizer.seen, eager.optimizer.seen)
            print(f"\nmasked rep {rep} use_graph={tr.use_graph}: bucket rel-L2 vs eager {e:.2e}")
            assert e < 1e-5, (rep, tr.use_graph, e)
            assert abs(float(o_e["loss"]) - float(o_g["loss"])) < 1e-6 * abs(float(o_e["loss"])) + 1e-7
        fused.optimizer_step(bs)
        e_f = _rel(fused.optimizer.seen, eager.optimizer.seen)
        print(f"masked fused micro-batches vs loop: bucket rel-L2 {e_f:.2e}")
        assert e_f < 5e-3
    # alternating masked / unmasked steps against a trainer that never sees a mask
    never = Stage1Trainer(step, params, accum=2, use_graph="step", optimizer=NoOpt())
    for rep in range(2):
        masked, plain = [batch(True), batch(True)], [batch(False), batch(False)]
        fused.optimizer_step(masked)
        assert float(fused.optimizer.seen.norm()) > 0
        o_f = fused.optimizer_step(plain)
        o_n = never.optimizer_step(plain)
        e = _rel(fused.optimizer.seen, never.optimizer.seen)
        print(f"unmasked step after a masked one vs a trainer without masks: loss {float(o_f['loss']):.8f} vs "
              f"{float(o_n['loss']):.8f}, bucket rel-L2 {e:.2e}")
        assert torch.equal(o_f["loss"], o_n["loss"]), rep
        assert e < 1e-5, (rep, e)
    bad = [batch(True), batch(False)]
    for tr in (eager, fused):
        with pytest.raises(ValueError, match="disagree"):
            tr.optimizer_step(bad)
