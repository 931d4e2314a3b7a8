"""Stage-1 training step (SURVEY.md section 8 row T1) on a B200: every backward kernel against torch.autograd of a
plain fp32 PyTorch restatement of the same op (attention: a float64 one), then the whole UNet's gradient w.r.t. the
layerwise context against autograd through the CPU oracle (oracle/unet_oracle.py, the pinned restatement of UNetModel.forward).
All calls go through the C ABI (adaprompt_b200.ops / adaprompt_b200.train -> ctypes -> libadaface_b200.so)."""
import contextlib
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DEV = "cuda"


def _rel(a, b):
    a, b = a.float().cpu(), b.float().cpu()
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


# ------------------------------------------------------------------------------------------------ bgemm
@pytest.mark.parametrize("M,N,K,nb0,nb1", [(256, 80, 48, 2, 3), (200, 136, 40, 1, 2), (80, 48, 256, 2, 2), (64, 64, 64, 1, 1)])
def test_bgemm_plain_strided(M, N, K, nb0, nb1):
    from adaprompt_b200 import ops
    a = _rand(nb0, M, nb1, K, seed=1, dtype=torch.bfloat16)           # [b0][row][b1][k]: head-sliced layout
    b = _rand(nb0, N, nb1, K, seed=2, dtype=torch.bfloat16)
    c = torch.full((nb0, nb1, M, N), 7.0, device=DEV, dtype=torch.float32)
    ops.bgemm(a, nb1 * K, (M * nb1 * K, K), b, nb1 * K, (N * nb1 * K, K), c, N, (nb1 * M * N, M * N), M=M, N=N, K=K,
              nb0=nb0, nb1=nb1, alpha=0.5)
    ref = 0.5 * torch.einsum("bmhk,bnhk->bhmn", a.float(), b.float())
    assert _rel(c, ref) < 1e-5


def test_bgemm_softmax_epilogues():
    from adaprompt_b200 import ops
    M, N, K, nb0, nb1, vr, vc = 192, 80, 48, 2, 2, 192, 77
    a = _rand(nb0, nb1, M, K, seed=3, dtype=torch.bfloat16)
    b = _rand(nb0, nb1, N, K, seed=4, dtype=torch.bfloat16)
    s = torch.einsum("bhmk,bhnk->bhmn", a.float(), b.float())
    rowv = _rand(nb0, nb1, M, seed=5)
    P = torch.empty(nb0, nb1, M, N, device=DEV, dtype=torch.bfloat16)
    sA, sB, sC = (nb1 * M * K, M * K), (nb1 * N * K, N * K), (nb1 * M * N, M * N)
    ops.bgemm(a, K, sA, b, K, sB, P, N, sC, M=M, N=N, K=K, nb0=nb0, nb1=nb1, mode=1, vec=rowv, sV=(nb1 * M, M),
              valid_rows=vr, valid_cols=vc)
    ref = torch.exp2(s - rowv[..., None])
    ref[..., vc:] = 0
    assert _rel(P, ref) < 4e-3
    # transposed problem with a column vector, then the dS epilogue on top of it
    Pt = torch.empty(nb0, nb1, N, M, device=DEV, dtype=torch.bfloat16)
    ops.bgemm(b, K, sB, a, K, sA, Pt, M, sC, M=N, N=M, K=K, nb0=nb0, nb1=nb1, mode=2, vec=rowv, sV=(nb1 * M, M),
              valid_rows=vc, valid_cols=vr)
    assert _rel(Pt, ref.transpose(2, 3)) < 4e-3
    dS = torch.empty(nb0, nb1, M, N, device=DEV, dtype=torch.float32)
    ops.bgemm(a, K, sA, b, K, sB, dS, N, sC, M=M, N=N, K=K, nb0=nb0, nb1=nb1, mode=3, vec=rowv, sV=(nb1 * M, M), P=P,
              ldp=N, sP=sC, valid_cols=vc, alpha=0.7)
    ref3 = 0.7 * P.float() * (s - rowv[..., None])
    ref3[..., vc:] = 0
    assert _rel(dS, ref3) < 1e-4
    dSt = torch.empty(nb0, nb1, N, M, device=DEV, dtype=torch.float32)
    ops.bgemm(b, K, sB, a, K, sA, dSt, M, sC, M=N, N=M, K=K, nb0=nb0, nb1=nb1, mode=4, vec=rowv, sV=(nb1 * M, M), P=Pt,
              ldp=M, sP=sC, valid_rows=vc, alpha=0.7)
    ref4 = 0.7 * Pt.float() * (s.transpose(2, 3) - rowv[:, :, None, :])
    ref4[:, :, vc:] = 0
    assert _rel(dSt, ref4) < 1e-4


# ------------------------------------------------------------------------------------------------ norms / activations
@pytest.mark.parametrize("B,HW,C,silu,eps", [(2, 256, 320, True, 1e-5), (3, 64, 1280, True, 1e-5), (2, 1024, 640, False, 1e-6),
                                             (1, 4096, 960, True, 1e-5)])
def test_groupnorm_backward(B, HW, C, silu, eps):
    from adaprompt_b200.train import GroupNormFn
    x = (_rand(B, HW, C, seed=1) * 2 + 0.3).requires_grad_(True)
    g, b = _rand(C, seed=2) * 0.5 + 1.0, _rand(C, seed=3) * 0.2
    dy = _rand(B, HW, C, seed=4, dtype=torch.bfloat16)
    y = GroupNormFn.apply(x, g, b, eps, silu)
    y.backward(dy)
    xr = x.detach().clone().requires_grad_(True)
    yr = F.group_norm(xr.permute(0, 2, 1), 32, g, b, eps).permute(0, 2, 1)
    if silu:
        yr = F.silu(yr)
    yr.backward(dy.float())
    assert _rel(y, yr) < 4e-3
    assert _rel(x.grad, xr.grad) < 2e-4


@pytest.mark.parametrize("rows,C,dt", [(512, 320, torch.bfloat16), (100, 1280, torch.bfloat16), (308, 768, torch.float32)])
def test_layernorm_backward_with_param_grads(rows, C, dt):
    from adaprompt_b200.train import LayerNormFn
    x = _rand(rows, C, seed=1).requires_grad_(True)
    g = (_rand(C, seed=2) * 0.5 + 1.0).requires_grad_(True)
    b = (_rand(C, seed=3) * 0.2).requires_grad_(True)
    dy = _rand(rows, C, seed=4, dtype=dt)
    LayerNormFn.apply(x, g, b, 1e-5, dt).backward(dy)
    xr, gr, br = (t.detach().clone().requires_grad_(True) for t in (x, g, b))
    F.layer_norm(xr, (C,), gr, br, 1e-5).backward(dy.float())
    assert _rel(x.grad, xr.grad) < 1e-4
    assert _rel(g.grad, gr.grad) < 1e-4
    assert _rel(b.grad, br.grad) < 1e-4


def test_geglu_and_quick_gelu_backward():
    from adaprompt_b200 import ops
    from adaprompt_b200.train import GegluFn
    proj = _rand(300, 2 * 640, seed=1, dtype=torch.bfloat16).requires_grad_(True)
    dh = _rand(300, 640, seed=2, dtype=torch.bfloat16)
    h = GegluFn.apply(proj)
    h.backward(dh)
    pr = proj.detach().float().requires_grad_(True)
    a, gate = pr.chunk(2, dim=-1)
    hr = a * F.gelu(gate)
    hr.backward(dh.float())
    assert _rel(h, hr) < 4e-3
    assert _rel(proj.grad, pr.grad) < 5e-3
    x = _rand(77, 3072, seed=3, dtype=torch.bfloat16)
    dy = _rand(77, 3072, seed=4, dtype=torch.bfloat16)
    xr = x.float().requires_grad_(True)
    yr = xr * torch.sigmoid(1.702 * xr)
    yr.backward(dy.float())
    assert _rel(ops.quick_gelu(x), yr) < 4e-3
    assert _rel(ops.quick_gelu(x, dy), xr.grad) < 5e-3


# ------------------------------------------------------------------------------------------------ linear / conv
def test_linear_dgrad_and_wgrad():
    from adaprompt_b200.train import linear
    T, K, N = 308, 768, 3072
    x = _rand(T, K, seed=1, dtype=torch.bfloat16).requires_grad_(True)
    w = (_rand(N, K, seed=2) * 0.05).requires_grad_(True)
    b = _rand(N, seed=3).requires_grad_(True)
    res = _rand(T, N, seed=5).requires_grad_(True)
    wb = w.detach().to(torch.bfloat16).contiguous()
    dy = _rand(T, N, seed=4)
    out = linear(x, wb, wb.t().contiguous(), b.detach(), residual=res, w_param=w, b_param=b)
    out.backward(dy)
    xr = x.detach().float().requires_grad_(True)
    wr = wb.float().requires_grad_(True)
    br, rr = b.detach().clone().requires_grad_(True), res.detach().clone().requires_grad_(True)
    (xr @ wr.t() + br + rr).backward(dy)
    assert _rel(x.grad, xr.grad) < 6e-3          # bf16 dY operand + bf16 result
    assert _rel(w.grad, wr.grad) < 6e-3
    assert _rel(b.grad, br.grad) < 1e-5
    assert torch.equal(res.grad, dy)


@pytest.mark.parametrize("kind,Cin,Cout,H", [("plain", 320, 640, 16), ("up", 640, 640, 8), ("down", 320, 320, 16)])
def test_conv_dgrad(kind, Cin, Cout, H):
    from adaprompt_b200.packing import pack_conv3x3
    from adaprompt_b200.train import Conv3x3Fn, DownsampleConvFn, UpsampleConvFn, _flip_conv_pack
    B = 2
    w = _rand(Cout, Cin, 3, 3, seed=1) * 0.05
    bias = _rand(Cout, seed=2)
    wb = w.to(torch.bfloat16).float()
    pk, pkb = pack_conv3x3(w), _flip_conv_pack(w)
    if kind == "plain":
        y = _rand(B, H, H, Cin, seed=3, dtype=torch.bfloat16).requires_grad_(True)
        out = Conv3x3Fn.apply(y, pk, pkb, bias, None, None)
        xr = y.detach().float().permute(0, 3, 1, 2).requires_grad_(True)
        ref = F.conv2d(xr, wb, bias, padding=1)
        leaf = y
    else:
        x = _rand(B, H, H, Cin, seed=3).requires_grad_(True)
        xr = x.detach().to(torch.bfloat16).float().permute(0, 3, 1, 2).requires_grad_(True)
        if kind == "up":
            out = UpsampleConvFn.apply(x, pk, pkb, bias)
            ref = F.conv2d(F.interpolate(xr, scale_factor=2, mode="nearest"), wb, bias, padding=1)
        else:
            out = DownsampleConvFn.apply(x, pk, pkb, bias)
            ref = F.conv2d(xr, wb, bias, stride=2, padding=1)
        leaf = x
    dy = _rand(*out.shape, seed=4)
    out.backward(dy)
    ref.backward(dy.to(torch.bfloat16).float().permute(0, 3, 1, 2))
    assert _rel(out, ref.permute(0, 2, 3, 1)) < 1e-4
    assert _rel(leaf.grad, xr.grad.permute(0, 2, 3, 1)) < (6e-3 if kind == "plain" else 1e-4)


def test_conv_out_dgrad():
    from adaprompt_b200 import ops
    B, H, C = 2, 16, 320
    w = _rand(4, C, 3, 3, seed=1) * 0.05
    dout = _rand(B, 4, H, H, seed=2)
    xr = torch.zeros(B, C, H, H, device=DEV, requires_grad=True)
    F.conv2d(xr, w, None, padding=1).backward(dout)
    assert _rel(ops.conv_out_dgrad(dout, w.contiguous(), C), xr.grad.permute(0, 2, 3, 1)) < 5e-3


# ------------------------------------------------------------------------------------------------ attention
# The attention backward has three implementations: the fused tcgen05 kernel (attention_bwd.cu: d = 40 / 80
# self-attention with N % 128 == 0), seven bgemm_kernel calls (bgemm.cu: every other UNet attention layer) and
# attention_small_bwd_kernel (train.cu: the CLIP text layers).  Each is compared with a float64 reference computed from
# the exact bf16 operands it reads, by global rel-L2, by its worst (sample, head, row) and by the exact zeros it owes.
LN2 = math.log(2.0)

# Limits (rel-L2, worst row) of dQ, dK, dV, each about 2x the worst value seen on one B200 (1000 W power limit) over
# the cases below.  Error sources:
#   FUSED_TOL (ops.attention_bwd with lse and delta from the reference): P and dS rounded to bf16 before the gradient
#     MMAs and the gradients stored as bf16, 2^-9 relative per element each.  Seen: rel 2.5e-3, rows 6.3e-3 (dQ),
#     5.0e-3 (dK), 4.6e-3 (dV), in every input regime.
#   COMPOSED_TOL (AttentionFn, fused and bgemm paths): in addition lse comes from the forward kernel, which sums the
#     bf16-rounded P (up to 2^-8 relative), and delta from the bf16 forward output O.  Seen: rel 3.1e-3 (dQ, dK),
#     2.4e-3 (dV); rows 7.6e-3, 7.0e-3, 4.1e-3, with random inputs and with dO = O + noise.
#   STRESS_TOL (AttentionFn with peaked softmax rows or dominant keys): dS = P o (dP - delta) cancels in the rows'
#     dominant entries, which turns the lse and delta errors above into larger relative errors of dQ and dK.  Seen:
#     rel 5.7e-3, 5.2e-3, 2.6e-3; rows 2.8e-2, 2.4e-2, 5.5e-3.
#   SMALL_TOL (attention_small_bwd_kernel: P and dS stay fp32 in shared memory): bf16 outputs only.  Seen: rel 1.7e-3,
#     rows 2.5e-3.
# In every random-input case _check_grads also shows each row limit to be below the worst-row error that one dropped
# 64-row block would cause (seen: at least 0.1).
FUSED_TOL = {"dQ": (5e-3, 1.3e-2), "dK": (5e-3, 1e-2), "dV": (5e-3, 1e-2)}
COMPOSED_TOL = {"dQ": (6e-3, 1.5e-2), "dK": (6e-3, 1.4e-2), "dV": (5e-3, 8e-3)}
STRESS_TOL = {"dQ": (1.2e-2, 6e-2), "dK": (1.1e-2, 5e-2), "dV": (5.5e-3, 1.1e-2)}
SMALL_TOL = {"dQ": (3.5e-3, 5e-3), "dK": (3.5e-3, 5e-3), "dV": (3.5e-3, 5e-3)}


def _attn_fwd64(qs, k, v):
    """O [B, Nq, h, d] = softmax(ln2 qs k^T) v in float64, one (sample, head) at a time."""
    B, Nq, h, d = qs.shape
    o = torch.empty(B, Nq, h, d, dtype=torch.float64, device=qs.device)
    for b in range(B):
        for j in range(h):
            s = (qs[b, :, j].double() @ k[b, :, j].double().t()) * LN2
            o[b, :, j] = torch.softmax(s, -1) @ v[b, :, j].double()
    return o


def _drop_block_sens(p, ds, q, k, g, ref):
    """Worst-row error (the row metric of _grad_errors) that a kernel would show if it dropped one 64-key block from dQ,
    or one 64-query block from one 128-key tile of dK / dV, of this (sample, head).  The smallest value over all blocks
    and tiles, so a row limit below it catches whichever block goes missing."""
    def terms(w, x):      # w [M, K] . x [K, d], its terms summed per 64-row block of x -> [M, ceil(K / 64), d]
        M, K = w.shape
        nb = (K + 63) // 64
        w = F.pad(w, (0, nb * 64 - K)).view(M, nb, 64).transpose(0, 1)
        x = F.pad(x, (0, 0, 0, nb * 64 - K)).view(nb, 64, -1)
        return torch.bmm(w, x).transpose(0, 1)

    def ratio(t, r):      # |dropped terms| of each row over the row's floor (see _grad_errors) -> [M, blocks]
        n = r.norm(dim=-1)
        return t.norm(dim=-1) / torch.maximum(n, n.pow(2).mean().sqrt())[:, None]

    def tiles(e):         # [keys, query blocks] -> smallest, over (128-key tile, query block), of the worst key in the tile
        nt = (e.shape[0] + 127) // 128
        return F.pad(e, (0, 0, 0, nt * 128 - e.shape[0])).view(nt, 128, -1).max(1).values.min().item()

    return {"dQ": ratio(LN2 * terms(ds, k), ref["dQ"]).max(0).values.min().item(),
            "dK": tiles(ratio(LN2 * terms(ds.t(), q), ref["dK"])),
            "dV": tiles(ratio(terms(p.t(), g), ref["dV"]))}


def _attn_bwd_ref(qs, k, v, dO, keep=False, sens=False):
    """Attention backward in float64 on the bf16 values the kernels read, one (sample, head) at a time on the inputs'
    device.  qs [B, Nq, h, d] carries d^-1/2 log2(e) (scores in the exp2 domain, as the projection packs fold it); k, v
    [B, nk, h, d] are the valid keys; dO [B, Nq, h, d].
      S = ln2 qs k^T   P = softmax(S)   O = P v   lse = log2 sum_j exp(S_j)   delta = rowsum(dO o O)
      dV = P^T dO      dS = P o (dO v^T - delta)      dQ = ln2 dS k      dK = ln2 dS^T qs
    Returns float64 O, dQ [B, Nq, h, d], dK, dV [B, nk, h, d], lse, delta [B, h, Nq]; keep: also P, dS [B, h, Nq, nk];
    sens: also _drop_block_sens of (sample 0, head 0)."""
    B, Nq, h, d = qs.shape
    nk = k.shape[1]
    f64 = dict(dtype=torch.float64, device=qs.device)
    r = {"O": torch.empty(B, Nq, h, d, **f64), "dQ": torch.empty(B, Nq, h, d, **f64),
         "dK": torch.empty(B, nk, h, d, **f64), "dV": torch.empty(B, nk, h, d, **f64),
         "lse": torch.empty(B, h, Nq, **f64), "delta": torch.empty(B, h, Nq, **f64)}
    if keep:
        r["P"], r["dS"] = torch.empty(B, h, Nq, nk, **f64), torch.empty(B, h, Nq, nk, **f64)
    for b in range(B):
        for j in range(h):
            q_, k_, v_, g_ = (t[b, :, j].double() for t in (qs, k, v, dO))
            s = (q_ @ k_.t()) * LN2
            lse = torch.logsumexp(s, -1)
            p = torch.exp(s - lse[:, None])
            del s
            o = p @ v_
            delta = (g_ * o).sum(-1)
            ds = p * (g_ @ v_.t() - delta[:, None])
            r["O"][b, :, j], r["lse"][b, j], r["delta"][b, j] = o, lse / LN2, delta
            r["dV"][b, :, j] = p.t() @ g_
            r["dQ"][b, :, j] = LN2 * (ds @ k_)
            r["dK"][b, :, j] = LN2 * (ds.t() @ q_)
            if keep:
                r["P"][b, j], r["dS"][b, j] = p, ds
            if sens and b == 0 and j == 0:
                r["sens"] = _drop_block_sens(p, ds, q_, k_, g_, {g: r[g][0, :, 0] for g in ("dQ", "dK", "dV")})
    return r


def _grad_errors(out, ref):
    """out, ref [B, rows, h, d] -> global rel-L2 and the worst row: the error of each (sample, row, head) over the larger
    of its reference norm and the RMS row norm of its (sample, head).  The floor keeps rows whose true gradient is ~0
    (saturated softmax rows, the first query of a causal layer) from turning rounding noise into large ratios."""
    diff = out.double() - ref
    n = ref.norm(dim=-1)
    floor = torch.maximum(n, n.pow(2).mean(dim=1, keepdim=True).sqrt()).clamp_min(1e-300)
    return {"rel": (diff.norm() / ref.norm()).item(), "row": (diff.norm(dim=-1) / floor).max().item()}


def _check_grads(label, got, ref, tol):
    """got / ref: dQ, dK, dV as [B, rows, h, d]; tol: (rel-L2, worst row) per gradient.  Prints the errors (and the
    sensitivities of ref, if it has them), asserts that each row limit is below its sensitivity, then the limits."""
    errs = {g: _grad_errors(got[g], ref[g]) for g in ("dQ", "dK", "dV")}
    sens = ref.get("sens")
    print(f"\n{label}: " + "  ".join(f"{g} rel {e['rel']:.2e} row {e['row']:.2e}" for g, e in errs.items())
          + ("  | one block dropped: " + " ".join(f"{g} {s:.2e}" for g, s in sens.items()) if sens else ""))
    if sens:
        for g, s in sens.items():
            assert tol[g][1] < s, f"{label}: the {g} row limit {tol[g][1]} would not catch a dropped block ({s:.3e})"
    for g, e in errs.items():
        assert e["rel"] < tol[g][0] and e["row"] < tol[g][1], (label, g, e)
    return errs


def _attn_bwd_inputs(B, Nq, nk, h, d, regime="random", seed=0):
    """bf16-exact float32 operands [B, n, h, d] (qs, k, v, dO) of one backward problem.  regime:
      random:   unit normal, qs scaled by d^-1/2 log2(e);
      peaked:   qs 8x larger: near one-hot softmax rows;
      dominant: the keys of the last 64-key block and of an even-indexed block scaled by 4, so that they carry most of
                each row's weight and reach the fused kernels through both stages of their two-stage ring;
      corr:     dO = O + 0.1 rms(O) noise: dP - delta cancels, which bf16 P / dS and delta make least accurate."""
    sc = d ** -0.5 * math.log2(math.e) * (8.0 if regime == "peaked" else 1.0)
    qs = (_rand(B, Nq, h, d, seed=seed) * sc).to(torch.bfloat16).float()
    k = _rand(B, nk, h, d, seed=seed + 1)
    if regime == "dominant":
        nb = (nk + 63) // 64
        for c in {nb - 1, (nb // 2) & ~1}:
            k[:, c * 64:(c + 1) * 64] *= 4.0
    k = k.to(torch.bfloat16).float()
    v = _rand(B, nk, h, d, seed=seed + 2, dtype=torch.bfloat16).float()
    g = _rand(B, Nq, h, d, seed=seed + 3)
    if regime == "corr":
        o = _attn_fwd64(qs, k, v).float()
        g = o + 0.1 * o.pow(2).mean().sqrt() * g
    return qs, k, v, g.to(torch.bfloat16).float()


def _rows_bf16(t, dp):
    """[B, n, h, d] -> bf16 [B*n, h*dp], each head's columns zero-padded to dp."""
    B, n, h, d = t.shape
    out = torch.zeros(B * n, h, dp, device=DEV, dtype=torch.bfloat16)
    out[..., :d] = t.reshape(B * n, h, d)
    return out.reshape(B * n, h * dp)


@contextlib.contextmanager
def _kernels():
    """Collects the names (spaces removed) of the CUDA kernels that ran inside the block."""
    names = []
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        yield names
        torch.cuda.synchronize()
    names.extend(e.key.replace(" ", "") for e in prof.key_averages())


def test_attention_backward_reference_matches_autograd():
    """_attn_bwd_ref against torch.autograd through softmax(ln2 q k^T) v, everything in float64."""
    B, N, nk, h, d = 2, 40, 24, 3, 8
    qs, k, v, g = (_rand(B, n, h, d, seed=s).double() for s, n in ((1, N), (2, nk), (3, nk), (4, N)))
    ref = _attn_bwd_ref(qs, k * 2, v, g, keep=True)
    qa, ka, va = (t.clone().requires_grad_(True) for t in (qs, k * 2, v))
    s = torch.einsum("bihd,bjhd->bhij", qa, ka) * LN2
    s.retain_grad()
    p = torch.softmax(s, -1)
    o = torch.einsum("bhij,bjhd->bihd", p, va)
    o.backward(g)
    for name, want in (("O", o), ("P", p), ("dS", s.grad), ("dQ", qa.grad), ("dK", ka.grad), ("dV", va.grad),
                       ("lse", torch.logsumexp(s, -1) / LN2), ("delta", (g * o).sum(-1).transpose(1, 2))):
        assert torch.allclose(ref[name], want.detach(), rtol=1e-12, atol=1e-12), name


FUSED_CASES = (
    [pytest.param(B, N, d, 8, "random", False, id=f"d{d}-B{B}-N{N}") for d in (40, 80)
     for B, N in ((2, 128), (3, 256), (3, 384), (1, 1024), (1, 2304), (1, 4096))]
    + [pytest.param(1, 9216, 40, 8, "random", False, id="d40-B1-N9216"),         # the 96x96 latent
       pytest.param(2, 256, 40, 1, "random", False, id="d40-B2-N256-h1"),
       pytest.param(1, 512, 80, 5, "random", False, id="d80-B1-N512-h5"),
       pytest.param(2, 1024, 40, 8, "random", True, id="d40-B2-N1024-qkview"),
       pytest.param(2, 512, 80, 8, "random", True, id="d80-B2-N512-qkview")]
    + [pytest.param(B, N, d, 8, regime, False, id=f"d{d}-B{B}-N{N}-{regime}") for regime in ("peaked", "dominant", "corr")
       for B, N, d in ((2, 128, 40), (1, 4096, 40), (2, 1024, 80), (1, 2304, 80))])


@pytest.mark.parametrize("B,N,d,heads,regime,qk_view", FUSED_CASES)
def test_attention_bwd_fused_kernel(B, N, d, heads, regime, qk_view):
    """ops.attention_bwd (its dQ and dK / dV kernels) with lse and delta taken from the reference, which keeps the
    forward and rowdot_heads out of the error: dQ, dK, dV against _attn_bwd_ref, the dQ / dK pad columns exactly 0.
    N = 128 is two key blocks, the depth of the ring; qk_view: Q and K are column views of one [tokens, Q|K] buffer."""
    from adaprompt_b200 import ops
    from adaprompt_b200.packing import head_pad
    dp = head_pad(d)
    qs, k, v, g = _attn_bwd_inputs(B, N, N, heads, d, regime, seed=N + d + heads)
    ref = _attn_bwd_ref(qs, k, v, g, sens=regime == "random")
    if qk_view:
        qk = torch.cat([_rows_bf16(qs, dp), _rows_bf16(k, dp)], 1)
        q, kk = qk[:, :heads * dp], qk[:, heads * dp:]
    else:
        q, kk = _rows_bf16(qs, dp), _rows_bf16(k, dp)
    vp, dop = _rows_bf16(v, dp), _rows_bf16(g, dp)
    qT, kT, dOT = (t.t().contiguous() for t in (q, kk, dop))
    dq, dk, dv = ops.attention_bwd(q, kk, vp, dop, qT, kT, dOT, ref["lse"].float(), ref["delta"].float(), B=B,
                                   heads=heads, N=N, d=d)
    dq, dk = dq.view(B, N, heads, dp), dk.view(B, N, heads, dp)
    assert not dq[..., d:].any() and not dk[..., d:].any(), "pad columns of dQ / dK"
    _check_grads(f"fused kernel B={B} N={N} d={d} heads={heads} {regime}" + (" [Q|K] views" if qk_view else ""),
                 {"dQ": dq[..., :d], "dK": dk[..., :d], "dV": dv.view(B, N, heads, d)}, ref, FUSED_TOL)


@pytest.mark.parametrize("bad", ["N64", "N192", "d160", "ld", "ldqt"])
def test_attention_bwd_rejects_bad_arguments(bad):
    """N not a positive multiple of 128, d = 160, a leading dimension that is not a multiple of 8 (16-byte TMA rows)
    and transposed operands narrower than B*N columns: ValueError, and no kernel runs."""
    from adaprompt_b200 import ops
    from adaprompt_b200.packing import head_pad
    B, h = 2, 8
    N = {"N64": 64, "N192": 192}.get(bad, 256)
    d = 160 if bad == "d160" else 40
    dp = head_pad(d)

    def z(*shape):
        return torch.zeros(*shape, device=DEV, dtype=torch.bfloat16)

    q = z(B * N, h * dp + 4)[:, :h * dp] if bad == "ld" else z(B * N, h * dp)
    k, vp, dop = z(B * N, h * dp), z(B * N, h * dp), z(B * N, h * dp)
    qT = z(h * dp, B * N - 8 if bad == "ldqt" else B * N)
    kT, dOT = z(h * dp, B * N), z(h * dp, B * N)
    lse, delta = torch.zeros(B, h, N, device=DEV), torch.zeros(B, h, N, device=DEV)
    torch.cuda.synchronize()
    with _kernels() as names:
        with pytest.raises(ValueError):
            ops.attention_bwd(q, k, vp, dop, qT, kT, dOT, lse, delta, B=B, heads=h, N=N, d=d)
    assert not any("attention_bwd_kernel" in n for n in names), names


def _attention_fn_grads(qs, k, v, g, nk_pad, fused, poison=False):
    """AttentionFn forward + backward on the UNet's buffers.  Self-attention (nk == nk_pad == N) takes q as the whole
    [tokens, Q|K] buffer and k as a view of its K half, as transformer_block_train does; cross-attention stores nk keys
    per sample with a stride of nk_pad rows.  fused = False sets ops.attention_bwd to None, which sends every shape down
    the bgemm path.  poison: key rows nk..nk_pad hold K values scaled by 2^10 and V values of +-2^100 instead of zeros.
    -> the gradients of q [B*N, ldq], k [B*nk_pad, h*dp], v [B*nk_pad, h*d]."""
    from adaprompt_b200 import ops
    from adaprompt_b200.packing import head_pad
    from adaprompt_b200.train import AttentionFn
    B, N, h, d = qs.shape
    nk = k.shape[1]
    dp = head_pad(d)
    kb = _rows_bf16(F.pad(k, (0, 0, 0, 0, 0, nk_pad - nk)), dp)
    vb = _rows_bf16(F.pad(v, (0, 0, 0, 0, 0, nk_pad - nk)), d)
    if poison:
        gen = torch.Generator().manual_seed(99)
        kb.view(B, nk_pad, -1)[:, nk:] = (torch.randn(B, nk_pad - nk, h * dp, generator=gen) * 1024).to(kb)
        sign = torch.randint(0, 2, (B, nk_pad - nk, h * d), generator=gen) * 2 - 1
        vb.view(B, nk_pad, -1)[:, nk:] = (sign * 2.0 ** 100).to(vb)
    if nk == nk_pad == N:
        qk = torch.cat([_rows_bf16(qs, dp), kb], 1)
        q, kk = qk.detach().requires_grad_(True), qk[:, h * dp:].detach().requires_grad_(True)
    else:
        q, kk = _rows_bf16(qs, dp).requires_grad_(True), kb.requires_grad_(True)
    vv = vb.requires_grad_(True)
    orig = ops.attention_bwd
    if not fused:
        ops.attention_bwd = None
    try:
        o = AttentionFn.apply(q, kk, vv, B, h, d, N, nk, nk_pad)
        o.backward(g.reshape(B * N, h * d).to(torch.bfloat16))
    finally:
        ops.attention_bwd = orig
    return q.grad, kk.grad, vv.grad


def _fused_eligible(N, nk, d):
    return d in (40, 80) and N == nk and N % 128 == 0


def _attention_fn_case(B, N, nk, d, regime="random", seed=1):
    """Forward + backward through AttentionFn against _attn_bwd_ref, on the fused path where the shape is eligible and
    always on the bgemm path (same inputs); every padding position of the gradients must be exactly 0."""
    from adaprompt_b200.packing import head_pad
    h, dp = 8, head_pad(d)
    nkp = (nk + 7) // 8 * 8
    qs, k, v, g = _attn_bwd_inputs(B, N, nk, h, d, regime, seed)
    ref = _attn_bwd_ref(qs, k, v, g, sens=regime == "random")
    for fused in ((True, False) if _fused_eligible(N, nk, d) else (False,)):
        dq, dk, dv = _attention_fn_grads(qs, k, v, g, nkp, fused)
        assert not dq[:, h * dp:].any(), "dq columns of the [Q|K] buffer outside the Q half"
        dq, dk, dv = dq[:, :h * dp].reshape(B, N, h, dp), dk.reshape(B, nkp, h, dp), dv.reshape(B, nkp, h, d)
        assert not dq[..., d:].any() and not dk[..., d:].any(), "pad columns of dQ / dK"
        assert not dk[:, nk:].any() and not dv[:, nk:].any(), "dK / dV rows of padded keys"
        _check_grads(f"AttentionFn {'fused' if fused else 'bgemm'} B={B} N={N} nk={nk} d={d} {regime}",
                     {"dQ": dq[..., :d], "dK": dk[:, :nk, :, :d], "dV": dv[:, :nk]}, ref,
                     STRESS_TOL if regime in ("peaked", "dominant") else COMPOSED_TOL)


def test_attention_backward_fused_qk_views_match_bgemm_path():
    """The layout the UNet trains with (q the whole [tokens, Q|K] buffer, k a column view of its K half) through both the
    fused kernel and the bgemm path, each against the float64 reference, at d = 40 and 80."""
    for d in (40, 80):
        _attention_fn_case(2, 512, 512, d, seed=11)


@pytest.mark.parametrize("B,N,nk,d", [(2, 256, 256, 40), (1, 1024, 1024, 80), (2, 64, 64, 160), (2, 512, 77, 40),
                                      (3, 256, 77, 80), (2, 64, 77, 160), (3, 1024, 1024, 40), (1, 4096, 4096, 40),
                                      (2, 2304, 2304, 80),
                                      # self-attention at the 64x64, 96x96 and 48x32 latents, 40x40 and 24x24 levels
                                      (1, 1536, 1536, 40), (2, 1600, 1600, 40),       # 1600 % 128 != 0: bgemm
                                      (2, 384, 384, 80), (2, 400, 400, 80), (1, 576, 576, 80),
                                      (2, 256, 256, 160), (2, 144, 144, 160), (3, 24, 24, 160),
                                      # cross-attention: 77 tokens at each level, and 2x / 3x KV multipliers
                                      (1, 4096, 77, 40), (1, 1024, 77, 80), (2, 256, 77, 160),
                                      (2, 256, 154, 80), (1, 1024, 231, 40)])
def test_attention_backward(B, N, nk, d):
    _attention_fn_case(B, N, nk, d)


@pytest.mark.parametrize("regime", ["peaked", "dominant", "corr"])
@pytest.mark.parametrize("B,N,nk,d", [(1, 1024, 1024, 40), (2, 256, 77, 80), (2, 144, 144, 160)])
def test_attention_backward_input_regimes(B, N, nk, d, regime):
    _attention_fn_case(B, N, nk, d, regime, seed=3)


@pytest.mark.parametrize("B,N,nk,d", [(2, 512, 77, 40), (2, 256, 154, 80), (2, 64, 77, 160), (1, 256, 231, 40)])
def test_attention_backward_garbage_pad_rows(B, N, nk, d):
    """Key rows nk..nk_pad are not attended: whatever they hold (K x 2^10, V = +-2^100), the gradients are bit-identical
    to those of zero pads, and the dK / dV rows of the pads are exactly 0."""
    nkp = (nk + 7) // 8 * 8
    qs, k, v, g = _attn_bwd_inputs(B, N, nk, 8, d, seed=5)
    clean = _attention_fn_grads(qs, k, v, g, nkp, fused=False)
    dirty = _attention_fn_grads(qs, k, v, g, nkp, fused=False, poison=True)
    for name, a, b in zip(("dq", "dk", "dv"), clean, dirty):
        assert torch.equal(a.view(torch.int16), b.view(torch.int16)), name
    assert not dirty[1].reshape(B, nkp, -1)[:, nk:].any() and not dirty[2].reshape(B, nkp, -1)[:, nk:].any()


@pytest.mark.parametrize("N", [256, 200])
@pytest.mark.parametrize("d", [40, 80, 160])
def test_rowdot_heads(N, d):
    """delta [B, heads, N] = sum_c dO[b, n, h*d + c] O[b, n, h*d + c].  Each bf16 x bf16 product is exact in fp32; the
    fp32 sum of d of them is within a few ulps of the sum of their magnitudes (seen: 6.6e-8 of it; limit 1.5e-7)."""
    from adaprompt_b200 import ops
    B, h = 3, 8
    a = _rand(B * N, h * d, seed=1, dtype=torch.bfloat16)
    b = _rand(B * N, h * d, seed=2, dtype=torch.bfloat16)
    delta = ops.rowdot_heads(a, b, B, N, h, d)
    prod = (a.double() * b.double()).view(B, N, h, d)
    err = ((delta.double() - prod.sum(-1).transpose(1, 2)).abs() / prod.abs().sum(-1).transpose(1, 2)).max().item()
    print(f"\nrowdot_heads N={N} d={d}: worst error over the sum of |terms| {err:.2e}")
    assert tuple(delta.shape) == (B, h, N) and err < 1.5e-7


def _attention_small_case(mult, B, causal, scale):
    """attention_small_bwd_kernel (the CLIP text layers, MKV multiplier mult) against float64 autograd: per-row errors on
    the q, k and v column blocks of dqkv; columns of a wider qkv buffer beyond q | k | v stay exactly 0."""
    from adaprompt_b200 import ops
    L, heads, E, extra = 77, 12, 768, 64
    k_off, v_off = E, E + E * mult
    ld = E + 2 * E * mult + extra
    qkv = _rand(B * L, ld, seed=mult + 4 * B, dtype=torch.bfloat16)
    dout = _rand(B * L, E, seed=9, dtype=torch.bfloat16)
    dqkv = ops.attention_small_bwd(qkv, dout, B=B, heads=heads, L=L, k_off=k_off, v_off=v_off, mult=mult, scale=scale,
                                   causal=causal)
    t = qkv.double().requires_grad_(True)
    q = t[:, :E].reshape(B, L, heads, 64)
    k = t[:, k_off:v_off].reshape(B, L, heads, mult, 64)
    v = t[:, v_off:v_off + E * mult].reshape(B, L, heads, mult, 64)
    s = torch.einsum("bihd,bjhrd->bhijr", q * scale, k)
    if causal:
        s = s.masked_fill(~torch.ones(L, L, device=DEV).tril().bool()[None, None, :, :, None], float("-inf"))
    p = torch.softmax(s.reshape(B, heads, L, L * mult), -1).reshape(B, heads, L, L, mult)
    o = torch.einsum("bhijr,bjhrd->bihd", p, v).reshape(B * L, E)
    o.backward(dout.double())
    fwd = torch.empty(B * L, E, device=DEV, dtype=torch.bfloat16)
    ops.attention_small(qkv, fwd, B=B, heads=heads, L=L, k_off=k_off, v_off=v_off, mult=mult, scale=scale, causal=causal)
    assert _rel(fwd, o) < 6e-3
    assert not dqkv[:, v_off + E * mult:].any(), "columns beyond q | k | v"

    def blocks(x):      # [B*L, ld] -> q, k, v blocks as [B, L, heads (x mult), 64]
        return {"dQ": x[:, :E].reshape(B, L, heads, 64), "dK": x[:, k_off:v_off].reshape(B, L, heads * mult, 64),
                "dV": x[:, v_off:v_off + E * mult].reshape(B, L, heads * mult, 64)}

    _check_grads(f"attention_small_bwd mult={mult} B={B} causal={causal} scale={scale}", blocks(dqkv), blocks(t.grad),
                 SMALL_TOL)


def test_attention_small_backward_mkv():
    """The text layers as the encoder runs them: causal, scale 1/8, one and two keys per token."""
    for mult in (1, 2):
        _attention_small_case(mult, 2, True, 0.125)


@pytest.mark.parametrize("mult,B,causal,scale", [(m, B, c, s) for m in (1, 2) for B in (1, 3) for c in (True, False)
                                                 for s in (0.125, 0.3)])
def test_attention_small_backward(mult, B, causal, scale):
    _attention_small_case(mult, B, causal, scale)


def test_attention_small_backward_rejects_mult_3():
    """Three keys per token need 295 KB of shared memory for a 77-token layer: ValueError, and the kernel does not run
    (the forward accepts up to 4)."""
    from adaprompt_b200 import ops
    B, L, E, mult = 1, 77, 768, 3
    qkv = torch.zeros(B * L, E + 2 * E * mult, device=DEV, dtype=torch.bfloat16)
    dout = torch.zeros(B * L, E, device=DEV, dtype=torch.bfloat16)
    torch.cuda.synchronize()
    with _kernels() as names:
        with pytest.raises(ValueError, match="shared memory"):
            ops.attention_small_bwd(qkv, dout, B=B, heads=12, L=L, k_off=E, v_off=E + E * mult, mult=mult)
    assert not any("attention_small_bwd_kernel" in n for n in names), names


def test_attention_backward_dispatch_runs_every_kernel():
    """Each backward kernel runs where it is meant to: the four attention_bwd_kernel instantiations on d = 40 / 80
    self-attention with N % 128 == 0 and no bgemm_kernel there; bgemm_kernel and no fused kernel everywhere else, each
    of its five modes at both tile widths (BN = 64 when the output has at most 64 columns); rowdot_heads_kernel on both
    paths; attention_small_bwd_kernel for the text layers."""
    from adaprompt_b200 import ops
    cases = [(1, 256, 256, 40), (1, 256, 256, 80), (2, 64, 64, 160), (1, 400, 400, 80), (1, 200, 200, 40),
             (1, 256, 77, 40)]
    seen = set()
    for B, N, nk, d in cases:
        qs, k, v, g = _attn_bwd_inputs(B, N, nk, 8, d, seed=2)
        with _kernels() as names:
            _attention_fn_grads(qs, k, v, g, (nk + 7) // 8 * 8, fused=True)
        fused = any("attention_bwd_kernel" in n for n in names)
        bgemm = any("bgemm_kernel" in n for n in names)
        print(f"\nbackward B={B} N={N} nk={nk} d={d}: fused kernel {fused}, bgemm {bgemm}")
        assert (fused, bgemm) == (_fused_eligible(N, nk, d), not _fused_eligible(N, nk, d)), (B, N, nk, d, names)
        assert any("rowdot_heads_kernel" in n for n in names)
        seen.update(names)
    qkv = _rand(77, 768 * 3, seed=1, dtype=torch.bfloat16)
    with _kernels() as names:
        ops.attention_small_bwd(qkv, _rand(77, 768, seed=2, dtype=torch.bfloat16), B=1, heads=12, L=77, k_off=768,
                                v_off=1536)
    seen.update(names)
    want = [f"attention_bwd_kernel<{d},{dkv}>" for d in (40, 80) for dkv in ("false", "true")]
    want += [f"bgemm_kernel<{bn},{m}>" for bn in (64, 128) for m in range(5)] + ["attention_small_bwd_kernel"]
    missing = [w for w in want if not any(w in n for n in seen)]
    assert not missing, (missing, sorted(n for n in seen if "bwd" in n or "bgemm" in n))


# ------------------------------------------------------------------------------------------------ whole UNet
def _unet():
    from adaprompt_b200.ldm_lite import SD15_UNET_CONFIG
    from adaprompt_b200.unet import UNetModel
    from adaprompt_b200.weights import spec_of, synth_state_dict
    with torch.device("meta"):
        unet = UNetModel(**SD15_UNET_CONFIG)
    unet = unet.to_empty(device=DEV)
    sd = synth_state_dict(spec_of(unet), 1234)
    unet.load_state_dict(sd)
    return unet.eval(), sd


def test_unet_context_gradient_matches_oracle_autograd():
    """d loss / d context of one distillation micro-step (batch 2, 32x32 latent) against autograd through the fp32
    CPU oracle.  Tolerance: 5e-2 relative L2 (bf16 operands through ~60 backward layers; the reference student runs
    TF32, main.py:815)."""
    from adaprompt_b200.train import distill_loss, unet_forward_train
    from oracle.golden_inputs import EXTRA_INFO
    from oracle.unet_oracle import UNetSpec, unet_forward
    unet, sd = _unet()
    g = torch.Generator().manual_seed(17)
    B = 2
    x = torch.randn(B, 4, 32, 32, generator=g)
    t = torch.tensor([501, 121])
    ctx = torch.randn(16 * B, 77, 768, generator=g)
    target = torch.randn(B, 4, 32, 32, generator=g)
    c_ref = ctx.clone().requires_grad_(True)
    eps_ref = unet_forward(sd, UNetSpec(), x, t, c_ref, dict(EXTRA_INFO))
    loss_ref = F.mse_loss(eps_ref, target)
    loss_ref.backward()
    c = ctx.to(DEV).requires_grad_(True)
    eps = unet_forward_train(unet, x.to(DEV), t.to(DEV), c, dict(EXTRA_INFO))
    loss = distill_loss(eps, target.to(DEV))
    loss.backward()
    assert _rel(eps, eps_ref) < 1e-2
    assert abs(loss.item() - loss_ref.item()) < 1e-2 * abs(loss_ref.item())
    err = _rel(c.grad, c_ref.grad)
    per_layer = [_rel(c.grad.reshape(B, 16, 77, 768)[:, l], c_ref.grad.reshape(B, 16, 77, 768)[:, l]) for l in range(16)]
    print("context grad rel-L2", err, "per layer", [f"{e:.3f}" for e in per_layer])
    # measured on B200: 9.2e-3 overall, 8e-3 .. 2.9e-2 per layer (bf16 operands through 25 blocks of backward): 2x that
    assert err < 2e-2 and max(per_layer) < 6e-2, (err, per_layer)


# ------------------------------------------------------------------------------------------------ conditioning half
def _clip_small(seed, layers, kv_mult=None):
    from adaprompt_b200.clip_text import CLIPTextConfigLite, CLIPTextModelWrapper
    from oracle import text_oracle as to
    sd = to.clip_synth_state_dict(seed, num_layers=layers, kv_mult=kv_mult)
    m = CLIPTextModelWrapper(CLIPTextConfigLite(num_hidden_layers=layers))
    if kv_mult:
        m.extend_clip_attention_MKV_multiplier(-1, -1, kv_mult[0], noise_std=0)
    m.load_state_dict(sd)
    return m.cuda(), sd


def _sbg_small(seed, layers, kv_mult=None, grad_scale=1.0):
    from adaprompt_b200.subj_basis_generator import SubjBasisGenerator
    from test_text_gpu import StubTokenizer
    m, sd = _clip_small(seed, layers, kv_mult)
    s = SubjBasisGenerator(num_out_embs_per_layer=16, clip_tokenizer=StubTokenizer(), prompt2token_proj_grad_scale=grad_scale)
    s.prompt2token_proj = m
    return s.cuda().train(), sd


def _cond_reference(sd_sbg, sd_frozen, hw, id_embs, tokens):
    from oracle import text_oracle as to
    subj, _ = to.subj_basis_generator_forward(sd_sbg, id_embs, hw, is_training=True)
    embedded = sd_frozen["text_model.embeddings.token_embedding.weight"][tokens]
    static, _, _ = to.splice_subject_embeddings(tokens, embedded, subj)
    return to.frozen_clip_encode(sd_frozen, tokens, static)


def _compare_param_grads(module, sd_ref, prefix="", tol=3e-2, skip=()):     # measured worst 1.3e-2 .. 1.5e-2
    worst = ("", 0.0)
    for name, p in module.named_parameters():
        ref = sd_ref[prefix + name].grad
        if name in skip or name.endswith("k_proj.bias"):
            continue   # softmax is invariant to a key bias (q.b is constant along a row): its true gradient is 0
        if ref is None or ref.abs().max() == 0:
            assert p.grad is None or p.grad.abs().max() == 0, name
            continue
        assert p.grad is not None, name
        e = _rel(p.grad, ref)
        if e > worst[1]:
            worst = (name, e)
        assert e < tol, (name, e)
    return worst


@pytest.mark.parametrize("kv_mult", [None, {0: 2, 1: 2, 2: 2}])
def test_conditioning_gradients_match_oracle_autograd(kv_mult):
    """SubjBasisGenerator (trainable CLIP text layers, MKV aware) -> splice -> frozen CLIP: every parameter gradient
    against autograd through the CPU oracle chain.  Tolerance 5e-2 relative L2 per parameter tensor."""
    from adaprompt_b200.train_cond import conditioning_train, sbg_forward_train
    from oracle import text_oracle as to
    sbg, sd_sbg = _sbg_small(21, 3, kv_mult)
    frozen, sd_frozen = _clip_small(22, 3)
    frozen.text_model.last_layers_skip_weights = [0.5, 0.5]
    for p in frozen.parameters():
        p.requires_grad = False
    g = torch.Generator().manual_seed(5)
    id_embs = torch.randn(2, 16, 768, generator=g) * 0.05
    tokens = torch.tensor([to.subject_prompt_ids(77), to.pad_ids([to.TOK_A, to.TOK_PHOTO]), to.subject_prompt_ids(77)])
    R = torch.randn(48, 77, 768, generator=g)
    # ---- reference
    sd_ref = {k: v.clone().requires_grad_(True) for k, v in sd_sbg.items()}
    hw_ref = torch.tensor([[1.0], [2.0], [4.0]], requires_grad=True)
    c_ref = _cond_reference(sd_ref, sd_frozen, hw_ref, id_embs, tokens)
    (c_ref * R).sum().backward()
    # ---- B200 path
    subj, _ = sbg_forward_train(sbg, id_embs.cuda())
    c = conditioning_train(frozen.text_model, tokens.cuda(), subj, to.TOK_Z)
    assert _rel(c, c_ref) < 1e-2
    (c * R.cuda()).sum().backward()
    worst = _compare_param_grads(sbg.prompt2token_proj, sd_ref, skip=("text_model.embeddings.token_embedding.weight",))
    tok_g = sbg.prompt2token_proj.text_model.embeddings.token_embedding.weight.grad
    tok_ref = sd_ref["text_model.embeddings.token_embedding.weight"].grad
    rows = tok_ref.abs().sum(1).nonzero().flatten()
    assert _rel(tok_g[rows.cuda()], tok_ref[rows]) < 5e-2 and float(tok_g.abs().sum()) > 0
    e_hw = _rel(sbg.hidden_state_layer_weights.grad, 5 * hw_ref.grad)       # grad scaler 5 (subj_basis_generator.py:580)
    print("worst parameter", worst, "hidden_state_layer_weights", e_hw)
    assert e_hw < 4e-2                                                       # measured 1.2e-2 .. 1.8e-2
    assert all(p.grad is None for p in frozen.parameters())


def test_distill_step_end_to_end_gradients():
    """Whole micro-step (configs[3] geometry scaled down: batch 2, 32x32 latent, 2-layer CLIPs): id embeddings ->
    SubjBasisGenerator -> splice -> frozen CLIP -> UNet -> MSE vs teacher eps; SubjBasisGenerator gradients against
    autograd through the CPU oracle chain (conditioning oracle + UNet oracle)."""
    from adaprompt_b200.train_cond import DistillStep, trainable_parameters
    from oracle import text_oracle as to
    from oracle.golden_inputs import EXTRA_INFO
    from oracle.unet_oracle import UNetSpec, make_alphas_cumprod, unet_forward
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
    step = DistillStep(unet, frozen.text_model, sbg, arc2face.eval(), StubTokenizer(), acp, to.TOK_Z)
    g = torch.Generator().manual_seed(9)
    B = 2
    batch = {"x0": torch.randn(B, 4, 32, 32, generator=g), "noise": torch.randn(B, 4, 32, 32, generator=g),
             "t": torch.tensor([601, 141]), "teacher_eps": torch.randn(B, 4, 32, 32, generator=g),
             "face_embs": F.normalize(torch.randn(B, 512, generator=g), dim=-1),
             "tokens": torch.tensor([to.subject_prompt_ids(77)] * B)}
    # ---- reference
    sd_ref = {k: v.clone().requires_grad_(True) for k, v in sd_sbg.items()}
    hw_ref = torch.tensor([[1.0], [2.0], [4.0]], requires_grad=True)
    with torch.no_grad():
        _, id_embs = to.arc2face_forward_face_embs(sd_arc, batch["face_embs"])
    c_ref = _cond_reference(sd_ref, sd_frozen, hw_ref, id_embs, batch["tokens"])
    a = acp[batch["t"]].view(-1, 1, 1, 1)
    x_noisy = a.sqrt() * batch["x0"] + (1 - a).sqrt() * batch["noise"]
    eps_ref = unet_forward(sd_unet, UNetSpec(), x_noisy, batch["t"], c_ref, dict(EXTRA_INFO))
    loss_ref = F.mse_loss(eps_ref, batch["teacher_eps"])
    loss_ref.backward()
    # ---- B200 path
    loss = step.micro_step({k: v.cuda() for k, v in batch.items()})
    assert abs(loss - loss_ref.item()) < 1e-2 * abs(loss_ref.item())
    scale = sbg.prompt2token_proj_grad_scale
    worst = ("", 0.0)
    for name, p in sbg.prompt2token_proj.named_parameters():
        ref = sd_ref[name].grad
        if name.endswith("token_embedding.weight") or name.endswith("k_proj.bias") or ref is None or ref.abs().max() == 0:
            continue
        e = _rel(p.grad / scale, ref)
        worst = max(worst, (name, e), key=lambda t: t[1])
    print("end-to-end worst parameter gradient error", worst, "n trainable", len(trainable_parameters(sbg)))
    assert worst[1] < 3e-2, worst                                            # measured 1.5e-2


def test_stage1_trainer_graph_matches_eager_and_steps_the_optimizer():
    """Stage1Trainer: (1) the CUDA-graph replay of the UNet forward + backward-to-context leaves the same gradient bucket
    as the eager tape (same kernels, same order: rel-L2 < 1e-5), twice in a row (replay with new inputs); (2) the bucket
    is what Prodigy consumes: the weights move, and the version-keyed packs of the inference mirror see the new
    weights (ADVICE r1: a stale bf16 pack after an optimizer step)."""
    from adaprompt_b200.train_cond import DistillStep, Stage1Trainer, trainable_parameters
    from oracle import text_oracle as to
    from oracle.unet_oracle import make_alphas_cumprod
    from test_text_gpu import StubTokenizer
    unet, _ = _unet()
    sbg, _ = _sbg_small(31, 2)
    frozen, _ = _clip_small(32, 2)
    arc2face, _ = _clip_small(33, 2)
    frozen.text_model.last_layers_skip_weights = [0.5, 0.5]
    for m in (frozen, arc2face):
        for p in m.parameters():
            p.requires_grad = False
    acp = torch.tensor(make_alphas_cumprod(), dtype=torch.float32)
    step = DistillStep(unet, frozen.text_model, sbg, arc2face.eval(), StubTokenizer(), acp, to.TOK_Z)
    params = trainable_parameters(sbg)
    g = torch.Generator().manual_seed(19)

    def batch():
        B = 2
        return {k: v.cuda() for k, v in {
            "x0": torch.randn(B, 4, 32, 32, generator=g), "noise": torch.randn(B, 4, 32, 32, generator=g),
            "t": torch.randint(0, 1000, (B,), generator=g), "teacher_eps": torch.randn(B, 4, 32, 32, generator=g),
            "face_embs": F.normalize(torch.randn(B, 512, generator=g), dim=-1),
            "tokens": torch.tensor([to.subject_prompt_ids(77)] * B)}.items()}

    class NoOpt:
        def step(self, flat):
            self.seen = flat.clone()

    eager = Stage1Trainer(step, params, accum=2, use_graph=False, optimizer=NoOpt())
    graph = Stage1Trainer(step, params, accum=2, use_graph=True, optimizer=NoOpt())      # UNet forward + backward graph
    whole = Stage1Trainer(step, params, accum=2, use_graph="step", optimizer=NoOpt())    # one graph per optimizer step,
    whole._gstep.fuse_unet = False                                                       # conditioning batched, UNet per micro-batch
    fused = Stage1Trainer(step, params, accum=2, use_graph="step", optimizer=NoOpt())    # + micro-batches fused through the UNet
    for rep in range(2):
        bs = [batch(), batch()]
        o_e = eager.optimizer_step(bs)
        for tr in (graph, whole):
            o_g = tr.optimizer_step(bs)
            # the scatter-add of the token-embedding gradient (index_add_, atomics) is the one non-deterministic sum
            assert _rel(tr.optimizer.seen, eager.optimizer.seen) < 1e-5, (rep, tr.use_graph)
            assert abs(float(o_e["loss"]) - float(o_g["loss"])) < 1e-6 * abs(float(o_e["loss"])) + 1e-7
            assert float(o_g["grad_norm"]) > 0 and float(tr.optimizer.seen.norm()) <= 0.5 + 1e-4      # clipped to 0.5
        # batch 2 x 2 as ONE UNet batch of 4: the same sums, but other tile schedules (split-K, tile width follow the row
        # count) re-associate the K sums and flip bf16 roundings downstream - the distance is that of two bf16 runs
        o_f = fused.optimizer_step(bs)
        e_f = _rel(fused.optimizer.seen, eager.optimizer.seen)
        print(f"fused micro-batches vs accumulation loop: gradient bucket rel-L2 {e_f:.2e}, loss "
              f"{float(o_f['loss']):.6f} vs {float(o_e['loss']):.6f}")
        assert e_f < 5e-3 and abs(float(o_e["loss"]) - float(o_f["loss"])) < 2e-4 * abs(float(o_e["loss"]))     # measured 2.2e-3, 4e-5
    # a prompt WITHOUT the placeholder passes through the splice untouched, with no host-side branch (and no sync)
    bs = [batch(), batch()]
    bs[0]["tokens"] = bs[0]["tokens"].clone()
    bs[0]["tokens"][1] = torch.tensor(to.subject_prompt_ids(77, placeholder=to.TOK_COMMA)).cuda()
    o_e = eager.optimizer_step(bs)
    o_g = whole.optimizer_step(bs)
    assert _rel(whole.optimizer.seen, eager.optimizer.seen) < 1e-5
    fused.optimizer_step(bs)
    assert _rel(fused.optimizer.seen, eager.optimizer.seen) < 5e-3
    # the real optimizer on the same bucket
    trainer = Stage1Trainer(step, params, accum=2, use_graph="step")
    w = sbg.prompt2token_proj.text_model.encoder.layers[0].mlp.fc1.weight
    layer = sbg.prompt2token_proj.text_model.encoder.layers[0]
    pack_before = layer.packed()["w1"].clone()
    w_before = w.detach().clone()
    for _ in range(3):
        trainer.optimizer_step([batch(), batch()])
    assert trainer.optimizer.param_groups[0]["k"] == 3
    assert not torch.equal(w.detach(), w_before)
    assert torch.equal(layer.packed()["w1"], w.detach().to(torch.bfloat16))          # repacked from the moved weights
    assert not torch.equal(layer.packed()["w1"], pack_before)


def test_multi_step_distillation_follows_the_reference_loop():
    """ddpm.py:2953-3039 with num_denoising_steps = 3, batch 2 (max_num_loss_steps = 3: every step counts; with batch 4 only
    the last step would): student inputs q_sample(pred_x0s[s-1], ts[s], noises[s]) - s = 0 wraps to the LAST teacher x0, as
    in the reference - targets = the teacher's noise predictions, loss = sum / sqrt(3); graph and eager paths agree; the
    gradient equals the hand-assembled sum of single-step gradients."""
    from adaprompt_b200.train import unet_forward_train, distill_loss
    from adaprompt_b200.train_cond import DistillStep, trainable_parameters
    from oracle import text_oracle as to
    from oracle.unet_oracle import make_alphas_cumprod
    from test_text_gpu import StubTokenizer
    unet, _ = _unet()
    sbg, _ = _sbg_small(41, 2)
    frozen, _ = _clip_small(42, 2)
    arc2face, _ = _clip_small(43, 2)
    frozen.text_model.last_layers_skip_weights = [0.5, 0.5]
    for m in (frozen, arc2face):
        for p in m.parameters():
            p.requires_grad = False
    acp = torch.tensor(make_alphas_cumprod(), dtype=torch.float32)
    g = torch.Generator().manual_seed(23)
    B, ND = 2, 3
    fixed = {"preds": [torch.randn(B, 4, 32, 32, generator=g).cuda() for _ in range(ND)],
             "x0s": [torch.randn(B, 4, 32, 32, generator=g).cuda() for _ in range(ND)],
             "noises": [torch.randn(B, 4, 32, 32, generator=g).cuda() for _ in range(ND)],
             "ts": [torch.tensor(v).cuda() for v in ([801, 640], [520, 410], [300, 222])]}

    class FakeTeacher:
        def __call__(self, ddpm, x_start, noise, t, context, num_denoising_steps=1):
            assert num_denoising_steps == ND and context.shape[1] == 21
            return fixed["preds"], fixed["x0s"], fixed["noises"], fixed["ts"]

    step = DistillStep(unet, frozen.text_model, sbg, arc2face.eval(), StubTokenizer(), acp, to.TOK_Z, teacher=FakeTeacher())
    params = trainable_parameters(sbg)
    batch = {k: v.cuda() for k, v in {
        "x0": torch.randn(B, 4, 32, 32, generator=g), "noise": torch.randn(B, 4, 32, 32, generator=g),
        "t": torch.tensor([801, 640]), "face_embs": F.normalize(torch.randn(B, 512, generator=g), dim=-1),
        "tokens": torch.tensor([to.subject_prompt_ids(77)] * B)}.items()}

    def grads_of(fn):
        for p in params:
            p.grad = None
        loss = fn()
        return float(loss), torch.cat([p.grad.reshape(-1) if p.grad is not None else torch.zeros_like(p).reshape(-1) for p in params])

    l_e, g_e = grads_of(lambda: step.multi_step_backward(batch, ND, use_graph=False))
    l_g, g_g = grads_of(lambda: step.multi_step_backward(batch, ND, use_graph=True))

    def by_hand():
        c = step.context(batch["face_embs"], batch["tokens"])
        total = 0
        for s in range(ND):
            x_s = step.q_sample(fixed["x0s"][s - 1], fixed["ts"][s], fixed["noises"][s])      # s = 0 -> x0s[-1]
            total = total + distill_loss(unet_forward_train(unet, x_s, fixed["ts"][s], c, dict(step.extra_info)), fixed["preds"][s])
        total = total / math.sqrt(ND)
        total.backward()
        return total.detach()

    l_h, g_h = grads_of(by_hand)
    assert abs(l_e - l_h) < 1e-6 * abs(l_h) and abs(l_g - l_h) < 1e-5 * abs(l_h)
    # graph path: the three per-step context gradients come back as separate tensors and are summed afterwards, the eager
    # tape accumulates them inside the bf16 dgrad chain: same values up to bf16 rounding of the accumulation order
    assert _rel(g_e, g_h) < 1e-5 and _rel(g_g, g_h) < 5e-3


# ------------------------------------------------------------------------------------------------ optimizer
@pytest.mark.parametrize("case", ["default", "decay_biascorr", "coupled_decay_growth"])
def test_prodigy_matches_reference_golden(case):
    """Fused flat-bucket Prodigy vs tests/golden/prodigy.pt (the UNMODIFIED ldm/prodigy.py run by
    oracle/make_golden_prodigy.py): 12 steps on a noisy quadratic, parameters and the adapted d."""
    import os
    from adaprompt_b200.prodigy import Prodigy
    g = torch.load(os.path.join(os.path.dirname(__file__), "golden", "prodigy.pt"))[case]
    params = [torch.nn.Parameter(t.clone().cuda()) for t in g["init"]]
    opt = Prodigy(params, lr=1.0, **g["kw"])
    for step, ns in enumerate(g["noises"]):
        for p, t, n in zip(params, g["targets"], ns):
            p.grad = (p.detach() - t.cuda()) + n.cuda()
        opt.step()
        assert abs(opt.param_groups[0]["d"] - g["d"][step]) <= 2e-4 * abs(g["d"][step]), (step, opt.param_groups[0]["d"], g["d"][step])
    for p, ref in zip(params, g["final"]):
        assert _rel(p, ref) < 1e-4


def test_distill_step_computes_teacher_eps_when_the_batch_has_none():
    """Row N4 wired into T1: without `teacher_eps` in the batch, DistillStep asks the Arc2Face teacher (a second UNet
    conditioned on the 21-token Arc2Face ID prompt, ddpm.py:5427,5451) for the target; the loss equals the one computed
    from the fp32 oracle's teacher prediction."""
    from adaprompt_b200.arc2face_teacher import Arc2FaceTeacher
    from adaprompt_b200.train_cond import DistillStep
    from oracle import text_oracle as to
    from oracle.golden_inputs import EXTRA_INFO
    from oracle.unet_oracle import UNetSpec, make_alphas_cumprod, unet_forward
    from test_text_gpu import StubTokenizer
    unet, sd_unet = _unet()
    sbg, sd_sbg = _sbg_small(31, 2)
    frozen, sd_frozen = _clip_small(32, 2)
    arc2face, sd_arc = _clip_small(33, 2)
    frozen.text_model.last_layers_skip_weights = [0.5, 0.5]
    acp = torch.tensor(make_alphas_cumprod(), dtype=torch.float32)
    step = DistillStep(unet, frozen.text_model, sbg, arc2face.eval(), StubTokenizer(), acp, to.TOK_Z,
                       teacher=Arc2FaceTeacher(unet))
    g = torch.Generator().manual_seed(19)
    B = 2
    batch = {"x0": torch.randn(B, 4, 32, 32, generator=g), "noise": torch.randn(B, 4, 32, 32, generator=g),
             "t": torch.tensor([451, 77]), "face_embs": F.normalize(torch.randn(B, 512, generator=g), dim=-1),
             "tokens": torch.tensor([to.subject_prompt_ids(77)] * B)}
    cuda = {k: v.cuda() for k, v in batch.items()}
    t_eps = step.teacher_eps(cuda["x0"], cuda["t"], cuda["noise"], cuda["face_embs"])
    with torch.no_grad():
        ctx21, _ = to.arc2face_forward_face_embs(sd_arc, batch["face_embs"], input_max_length=21)
        a = acp[batch["t"]].view(-1, 1, 1, 1)
        x_noisy = a.sqrt() * batch["x0"] + (1 - a).sqrt() * batch["noise"]
        t_ref = unet_forward(sd_unet, UNetSpec(), x_noisy, batch["t"], ctx21.repeat_interleave(16, 0), dict(EXTRA_INFO))
    assert tuple(ctx21.shape) == (B, 21, 768)
    e = _rel(t_eps, t_ref)
    print(f"teacher eps rel-L2 {e:.3e}")
    assert e < 1e-2
    for p in unet.parameters():                      # Arc2FaceTeacher froze the shared UNet: the student path needs no weight grads either
        assert not p.requires_grad
    loss = step.micro_step(cuda)
    assert loss > 0 and all(torch.isfinite(p.grad).all() for p in sbg.prompt2token_proj.parameters() if p.grad is not None)
