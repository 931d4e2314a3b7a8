"""CPU checks of tests/norm_reference.py: the float64 GroupNorm / LayerNorm references against torch's float64
group_norm / layer_norm and autograd, the metrics, the input regimes and the defect models.  No GPU needed."""
import pytest
import torch
import torch.nn.functional as F

import norm_reference as nr


def _d(*shape, seed):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed), dtype=torch.float64)


def _torch_gn(x, gamma, beta, eps, silu):
    y = F.group_norm(x.permute(0, 2, 1), 32, gamma, beta, eps).permute(0, 2, 1)
    return F.silu(y) if silu else y


@pytest.mark.parametrize("B,HW,C0,C1,silu,eps", [(2, 15, 640, 320, True, 1e-5), (1, 7, 128, 0, False, 1e-6),
                                                 (3, 1, 256, 256, True, 1e-5)])
def test_gn_ref_matches_torch(B, HW, C0, C1, silu, eps):
    x0, x1 = _d(B, HW, C0, seed=1) * 2 + 0.3, (_d(B, HW, C1, seed=2) - 0.5) if C1 else None
    C = C0 + C1
    gamma, beta = 1 + 0.1 * _d(C, seed=3), 0.1 * _d(C, seed=4)
    y, mean, rstd = nr.gn_ref(x0, x1, gamma, beta, eps, silu)
    x = x0 if x1 is None else torch.cat([x0, x1], -1)
    assert torch.allclose(y, _torch_gn(x, gamma, beta, eps, silu), rtol=1e-12, atol=1e-12)
    g = x.reshape(B, HW, 32, C // 32)
    assert torch.allclose(mean, g.mean(dim=(1, 3)), rtol=1e-12, atol=1e-14)
    assert torch.allclose(rstd, (g.var(dim=(1, 3), unbiased=False) + eps).rsqrt(), rtol=1e-12)


@pytest.mark.parametrize("silu,dres", [(True, True), (False, False), (True, False)])
def test_gn_bwd_ref_matches_autograd(silu, dres):
    B, HW, C, eps = 2, 9, 320, 1e-5
    x = (_d(B, HW, C, seed=5) * 1.5 + 0.2).requires_grad_(True)
    gamma, beta = 1 + 0.2 * _d(C, seed=6), 0.3 * _d(C, seed=7)
    dy, r = _d(B, HW, C, seed=8), (_d(B, HW, C, seed=9) if dres else None)
    _torch_gn(x, gamma, beta, eps, silu).backward(dy)
    mean, rstd = nr.gn_stats_ref(x.detach(), eps)
    dx = nr.gn_bwd_ref(x.detach(), mean, rstd, gamma, beta, silu, dy, r)
    assert torch.allclose(dx, x.grad + (r if dres else 0), rtol=1e-10, atol=1e-12)
    assert nr.gn_bwd_ref(x.detach(), mean, rstd, gamma, beta, silu, dy, r, drop_rows=slice(0, 0)).equal(dx)


@pytest.mark.parametrize("rows,C", [(1, 4), (7, 388), (3, 2048)])
def test_ln_ref_matches_torch_and_autograd(rows, C):
    eps = 1e-5
    x = (_d(rows, C, seed=1) * 1.7 + 0.2).requires_grad_(True)
    gamma = (1 + 0.1 * _d(C, seed=2)).requires_grad_(True)
    beta = (0.1 * _d(C, seed=3)).requires_grad_(True)
    dy, dres = _d(rows, C, seed=4), _d(rows, C, seed=5)
    yt = F.layer_norm(x, (C,), gamma, beta, eps)
    yt.backward(dy)
    y, mean, rstd = nr.ln_ref(x.detach(), gamma.detach(), beta.detach(), eps)
    assert torch.allclose(y, yt.detach(), rtol=1e-12, atol=1e-12)
    assert torch.allclose(mean, x.detach().mean(-1), atol=1e-14)
    dx, dg, db = nr.ln_bwd_ref(x.detach(), gamma.detach(), eps, dy, dres)
    assert torch.allclose(dx, x.grad + dres, rtol=1e-10, atol=1e-12)
    assert torch.allclose(dg, gamma.grad, rtol=1e-10, atol=1e-12)
    assert torch.allclose(db, beta.grad, rtol=1e-10, atol=1e-12)


def test_metrics_see_one_group_and_one_row():
    """A 2 % error in one of 64 (sample, group) pairs moves global rel-L2 by ~2.5e-3 but the worst-group metric by 2e-2;
    likewise for one row of 64."""
    ref = _d(2, 100, 320, seed=1)
    got = ref.clone()
    got[1, :, 40:50] *= 1.02
    assert nr.rel_l2(got, ref) < 3e-3
    assert abs(nr.worst_group(got, ref) - 0.02) < 1e-3
    rows = _d(64, 256, seed=2)
    got = rows.clone()
    got[17] *= 1.02
    assert nr.rel_l2(got, rows) < 3e-3 and abs(nr.worst_row(got, rows) - 0.02) < 1e-3
    # the floor: an all-zero group is judged against the RMS group norm of its sample, not against zero
    ref[0, :, :10] = 0
    got = ref.clone()
    got[0, :, :10] = 1e-9
    assert nr.worst_group(got, ref) < 2e-9


def test_stats_errors_units():
    mean, rstd = _d(2, 32, seed=1), _d(2, 32, seed=2).abs() + 0.5
    mr = nr.stats_as_mr(mean, rstd)
    assert mr.dtype == torch.float32 and mr.shape == (128,)
    e = nr.stats_errors(mr, mean, rstd)
    assert e["mean"] < 1e-6 and e["rstd"] < 1e-7
    shifted = mr.double().reshape(2, 32, 2).clone()
    shifted[1, 5, 0] += 0.01 / rstd[1, 5]
    shifted[0, 3, 1] *= 1.003
    e = nr.stats_errors(shifted, mean, rstd)
    assert abs(e["mean"] - 0.01) < 1e-6 and abs(e["rstd"] - 0.003) < 1e-7


def test_slot_bounds_leave_trailing_slots_empty():
    b = nr.slot_bounds(1000, 62)
    assert b[0] == (0, 17) and b[58] == (986, 1000) and b[59:] == [(1000, 1000)] * 3
    assert nr.slot_bounds(1, 1) == [(0, 1)]


def test_regimes():
    B, HW, C = 2, 100, 320
    x = nr.gn_input("structured", B, HW, C, 1)
    assert x.dtype == torch.float32 and x.shape == (B, HW, C)
    mean, rstd = nr.gn_stats_ref(x, 0.0)
    assert (mean.abs() * rstd).max() < 3             # iid-level accuracy applies: no large mean/std
    assert len(set(torch.round(mean[0], decimals=3).tolist())) == 32
    assert torch.all(rstd[0] > 1.2 * rstd[1])        # per-sample scale
    for k in (30, 100, 300):
        mean, rstd = nr.gn_stats_ref(nr.gn_input(f"offset{k}", B, HW, C, 1), 0.0)
        ratio = mean.abs() * rstd
        assert ratio.min() > 0.8 * k and ratio.max() < 1.2 * k
    x = nr.gn_input("degenerate", B, HW, C, 1)
    assert torch.all(x[:, :, :10] == 0) and torch.all(x[:, :, 10:20] == -0.75) and x[:, 50, 20].eq(1e4).all()
    rows = nr.ln_input("offset1000", 9, 640, 1)
    _, m, r = nr.ln_ref(rows, torch.ones(640), torch.zeros(640), 0.0)
    assert ((m * r - 1000).abs() < 200).all()


def test_defect_models_are_visible():
    """The defect models change what they model and nothing else: no defect applies where it cannot happen."""
    x = nr.gn_input("structured", 2, 1000, 320, 1)
    g, b = nr.affine(320, 2)
    sens = nr.gn_output_sensitivity(x, g, b, 1e-5, True, 62)
    assert set(sens) == {"drop_slot", "next_sample", "neighbour"} and min(sens.values()) > 0.05
    assert set(nr.gn_output_sensitivity(x[:1, :15], g, b, 1e-5, True, 1)) == {"neighbour"}
    mean, rstd = nr.gn_stats_ref(x, 1e-5)
    dy = nr.gn_input("structured", 2, 1000, 320, 5).bfloat16()
    sens = nr.gn_bwd_sensitivity(x, mean, rstd, g, b, False, dy, 62)
    assert set(sens) == {"drop_chunk", "next_sample", "neighbour"} and min(sens.values()) > 0.05
    rows = nr.ln_input("structured", 7, 388, 1)
    g, b = nr.affine(388, 2)
    assert min(nr.ln_sensitivity(rows, g, b, 1e-5).values()) > 0.05
    assert min(nr.ln_bwd_sensitivity(rows, g, 1e-5, nr.ln_input("structured", 7, 388, 5)).values()) > 0.05
