"""Float64 references of GroupNorm(32) [+SiLU] and LayerNorm, forward and backward, the error metrics the norm tests
use, the input regimes they draw from, and the bookkeeping defects their limits must be able to see.

Everything here is plain torch and runs on whatever device its inputs live on: on the CPU in
tests/test_norm_reference.py (checked against torch's float64 group_norm / layer_norm and autograd), on the GPU in
tests/test_norm_gpu.py.  References are computed in float64 from the exact fp32 / bf16 values the kernel received."""
import torch

GROUPS = 32


# ------------------------------------------------------------------------------------------------ references
def _silu_grad(z):
    s = torch.sigmoid(z)
    return s * (1 + z * (1 - s))


def _per_channel(v, cpg):
    """[B, 32] -> [B, 1, C]: each group's value repeated over its channels."""
    return v.repeat_interleave(cpg, dim=1)[:, None, :]


def gn_stats_ref(x, eps):
    """x [B, HW, C] -> (mean, rstd) [B, 32] in float64."""
    x = x.double()
    B, HW, C = x.shape
    g = x.reshape(B, HW, GROUPS, C // GROUPS)
    mean = g.mean(dim=(1, 3))
    var = (g - mean[:, None, :, None]).pow(2).mean(dim=(1, 3))
    return mean, (var + eps).rsqrt()


def gn_apply_ref(x, mean, rstd, gamma, beta, silu):
    """y = silu?((x - mean) * rstd * gamma + beta) with the given per-(sample, group) statistics, float64."""
    x = x.double()
    cpg = x.shape[-1] // GROUPS
    z = (x - _per_channel(mean.double(), cpg)) * _per_channel(rstd.double(), cpg) * gamma.double() + beta.double()
    return z * torch.sigmoid(z) if silu else z


def gn_ref(x0, x1, gamma, beta, eps, silu):
    """GroupNorm(32) [+SiLU] of the channel concat [x0 | x1] (x1 may be None): y [B, HW, C], mean and rstd [B, 32]."""
    x = x0 if x1 is None else torch.cat([x0, x1], -1)
    mean, rstd = gn_stats_ref(x, eps)
    return gn_apply_ref(x, mean, rstd, gamma, beta, silu), mean, rstd


def gn_bwd_ref(x, mean, rstd, gamma, beta, silu, dy, dres=None, drop_rows=None):
    """Analytic backward of y = silu?(xhat * gamma + beta), xhat = (x - mean) * rstd, with mean / rstd those of the
    group (taken as given, so a test can feed the kernel the same values):
        dxhat = dy * silu'(z) * gamma;  dx = rstd * (dxhat - mean_g(dxhat) - xhat * mean_g(dxhat * xhat)) (+ dres).
    drop_rows: a slice of pixels whose contribution to the two group means is left out (a defect model)."""
    x, dy = x.double(), dy.double()
    B, HW, C = x.shape
    cpg = C // GROUPS
    m, r = _per_channel(mean.double(), cpg), _per_channel(rstd.double(), cpg)
    xh = (x - m) * r
    g = gamma.double()
    dz = dy * _silu_grad(xh * g + beta.double()) if silu else dy
    d = dz * g
    d_in, p_in = d, d * xh
    if drop_rows is not None:
        d_in, p_in = d_in.clone(), p_in.clone()
        d_in[:, drop_rows] = 0
        p_in[:, drop_rows] = 0
    n = HW * cpg
    m1 = _per_channel(d_in.reshape(B, HW, GROUPS, cpg).sum(dim=(1, 3)) / n, cpg)
    m2 = _per_channel(p_in.reshape(B, HW, GROUPS, cpg).sum(dim=(1, 3)) / n, cpg)
    dx = r * (d - m1 - xh * m2)
    return dx if dres is None else dx + dres.double()


def ln_ref(x, gamma, beta, eps):
    """LayerNorm over the last dim in float64: y, mean and rstd [rows]."""
    x = x.double()
    mean = x.mean(-1)
    var = (x - mean[..., None]).pow(2).mean(-1)
    rstd = (var + eps).rsqrt()
    return (x - mean[..., None]) * rstd[..., None] * gamma.double() + beta.double(), mean, rstd


def ln_bwd_ref(x, gamma, eps, dy, dres=None):
    """Analytic LayerNorm backward in float64: dx (+ dres), dgamma = sum_rows dy * xhat, dbeta = sum_rows dy."""
    x, dy = x.double(), dy.double()
    _, mean, rstd = ln_ref(x, torch.ones_like(gamma), torch.zeros_like(gamma), eps)
    xh = (x - mean[..., None]) * rstd[..., None]
    d = dy * gamma.double()
    dx = rstd[..., None] * (d - d.mean(-1, keepdim=True) - xh * (d * xh).mean(-1, keepdim=True))
    if dres is not None:
        dx = dx + dres.double()
    rows = dy.reshape(-1, dy.shape[-1])
    return dx, (rows * xh.reshape(rows.shape)).sum(0), rows.sum(0)


# ------------------------------------------------------------------------------------------------ metrics
def rel_l2(got, ref):
    ref = ref.double()
    return ((got.double() - ref).norm() / ref.norm().clamp_min(1e-300)).item()


def _worst(diff, ref, dims):
    """Worst ratio of a block's error norm to the larger of its reference norm and the RMS block norm of its sample.
    The floor keeps blocks whose true value is ~0 (an all-zero group, a row of zero gradient) from turning rounding
    noise into large ratios.  diff / ref: [S, blocks, ...] with the block's elements in `dims`."""
    n = ref.norm(dim=dims) if dims else ref.abs()
    floor = torch.maximum(n, n.pow(2).mean(dim=1, keepdim=True).sqrt()).clamp_min(1e-300)
    e = diff.norm(dim=dims) if dims else diff.abs()
    return (e / floor).max().item()


def worst_group(got, ref):
    """Worst (sample, group) rel-L2 of [B, HW, C] tensors, floored at the RMS group norm of the sample."""
    B, HW, C = ref.shape
    ref = ref.double().reshape(B, HW, GROUPS, C // GROUPS).transpose(1, 2)
    diff = got.double().reshape(B, HW, GROUPS, C // GROUPS).transpose(1, 2) - ref
    return _worst(diff, ref, (2, 3))


def worst_row(got, ref):
    """Worst row rel-L2 of [rows, C] tensors (one sample), floored at the RMS row norm."""
    ref = ref.double().reshape(1, -1, ref.shape[-1])
    return _worst(got.double().reshape(ref.shape) - ref, ref, (2,))


def stats_errors(mr, mean, rstd):
    """mr: kernel statistics [B*32*2] or [B, 32, 2] (mean, rstd interleaved) against float64 mean / rstd [B, 32]:
    the worst mean error in units of the group's sqrt(var + eps) and the worst relative rstd error."""
    mr = mr.double().reshape(mean.shape[0], GROUPS, 2)
    rstd = rstd.double()
    return {"mean": ((mr[..., 0] - mean.double()).abs() * rstd).max().item(),
            "rstd": (mr[..., 1] / rstd - 1).abs().max().item()}


def stats_as_mr(mean, rstd):
    """Float64 statistics -> the kernel's fp32 mean_rstd layout [B*32*2]."""
    return torch.stack([mean, rstd], -1).float().reshape(-1).contiguous()


# ------------------------------------------------------------------------------------------------ input regimes
def _randn(shape, gen, device):
    return torch.randn(*shape, generator=gen, dtype=torch.float64).to(device)


def _ramp(n, steep=6.0):
    """Increasing convex ramp over n positions, zero mean, unit RMS: the last positions hold the largest values, so
    leaving the last slot, chunk or vector out of a statistic changes it visibly."""
    if n == 1:
        return torch.zeros(1, dtype=torch.float64)
    r = torch.expm1(steep * torch.linspace(0, 1, n, dtype=torch.float64))
    r = r - r.mean()
    return r / r.pow(2).mean().sqrt()


def gn_input(regime, B, HW, C, seed=0, device="cpu"):
    """fp32 [B, HW, C] GroupNorm input.  regime:
      iid:        2 * randn + 0.3;
      structured: per-sample scale (1 + 0.5 b) times (a distinct offset per group and per channel + a convex per-pixel
                  ramp + noise): every slot, channel and sample contributes a distinguishable amount;
      offset30, offset100, offset300: each group's mean is k times its std (std 0.5..2 by group, sign alternating);
      degenerate: iid, except in every sample group 0 is all zero, group 1 is the constant -0.75 (variance 0 < eps)
                  and group 2 has a single 1e4 outlier pixel."""
    gen = torch.Generator().manual_seed(seed)
    cpg = C // GROUPS
    z = _randn((B, HW, C), gen, "cpu")
    if regime == "iid":
        x = 2 * z + 0.3
    elif regime == "structured":
        goff = 2 * torch.linspace(-1, 1, GROUPS, dtype=torch.float64)[torch.randperm(GROUPS, generator=gen)]
        coff = goff.repeat_interleave(cpg) + 0.3 * _randn((C,), gen, "cpu")
        scale = 1 + 0.5 * torch.arange(B, dtype=torch.float64)
        x = scale[:, None, None] * (coff + _ramp(HW)[:, None] + 0.5 * z)
    elif regime.startswith("offset"):
        k = float(regime[6:])
        std = torch.logspace(-1, 1, GROUPS, base=2, dtype=torch.float64)
        sign = torch.tensor([1.0, -1.0], dtype=torch.float64).repeat(GROUPS // 2)
        x = (std * (k * sign)).repeat_interleave(cpg) + std.repeat_interleave(cpg) * z
    elif regime == "degenerate":
        x = 2 * z + 0.3
        x[:, :, :cpg] = 0
        x[:, :, cpg:2 * cpg] = -0.75
        x[:, HW // 2, 2 * cpg] = 1e4
    else:
        raise ValueError(regime)
    return x.float().to(device)


def ln_input(regime, rows, C, seed=0, device="cpu"):
    """fp32 [rows, C] LayerNorm input.  iid: 1.7 randn + 0.2; structured: per-row scale and shift times (distinct
    per-channel offsets + a convex ramp over the channels + noise); offsetK: row mean K times the row std."""
    gen = torch.Generator().manual_seed(seed)
    z = _randn((rows, C), gen, "cpu")
    if regime == "iid":
        x = 1.7 * z + 0.2
    elif regime == "structured":
        r = torch.arange(rows, dtype=torch.float64)[:, None]
        x = (1 + 0.15 * (r % 7)) * (0.5 * _randn((C,), gen, "cpu") + _ramp(C, 12.0) + 0.5 * z) + 0.3 * (r % 5 - 2)
    elif regime.startswith("offset"):
        k = float(regime[6:])
        std = torch.logspace(-1, 1, rows, base=2, dtype=torch.float64)[:, None]
        x = std * (k + z)
    else:
        raise ValueError(regime)
    return x.float().to(device)


def affine(C, seed, device="cpu"):
    """gamma = 1 + 0.1 randn, beta = 0.1 randn (fp32)."""
    gen = torch.Generator().manual_seed(seed)
    g = 1 + 0.1 * torch.randn(C, generator=gen)
    b = 0.1 * torch.randn(C, generator=gen)
    return g.to(device), b.to(device)


# ------------------------------------------------------------------------------------------------ defect models
def slot_bounds(HW, slots):
    """Pixel ranges [p0, p1) of the slots (or chunks) the kernels cut a sample into: ceil(HW / slots) pixels each, the
    last ones short or empty."""
    per = (HW + slots - 1) // slots
    return [(min(HW, s * per), min(HW, (s + 1) * per)) for s in range(slots)]


def gn_stats_defects(x, eps, slots):
    """Statistics [B, 32] that plausible bookkeeping defects would produce, as {name: (mean, rstd)}:
      drop_slot:  the last non-empty slot left out of the fold (only with more than one slot);
      neighbour:  not a statistic but a channel map (see gn_defect_outputs);
      next_sample: sample b gets sample b+1's statistics (only with B > 1)."""
    x = x.double()
    B, HW, C = x.shape
    out = {}
    bounds = [b for b in slot_bounds(HW, slots) if b[1] > b[0]]
    if len(bounds) > 1:
        p0, p1 = bounds[-1]
        keep = torch.cat([x[:, :p0], x[:, p1:]], 1)
        out["drop_slot"] = gn_stats_ref(keep, eps)
    mean, rstd = gn_stats_ref(x, eps)
    if B > 1:
        out["next_sample"] = (mean.roll(-1, 0), rstd.roll(-1, 0))
    return out


def gn_defect_outputs(x, gamma, beta, eps, silu, slots):
    """GroupNorm outputs under each defect: {name: y}, including `neighbour`, where the last channel of every group
    (but the last) takes the next group's statistics."""
    mean, rstd = gn_stats_ref(x, eps)
    ys = {k: gn_apply_ref(x, m, r, gamma, beta, silu) for k, (m, r) in gn_stats_defects(x, eps, slots).items()}
    B, HW, C = x.shape
    cpg = C // GROUPS
    y = gn_apply_ref(x, mean, rstd, gamma, beta, silu)
    last = torch.arange(cpg - 1, C - cpg, cpg)
    mn, rn = _per_channel(mean, cpg)[..., last + cpg], _per_channel(rstd, cpg)[..., last + cpg]
    z = (x.double()[..., last] - mn) * rn * gamma.double()[last] + beta.double()[last]
    y[..., last] = z * torch.sigmoid(z) if silu else z
    ys["neighbour"] = y
    return ys


def gn_stats_sensitivity(x, eps, slots):
    """{defect: stats_errors of its statistics against the true ones}: what the statistics limits must stay below."""
    mean, rstd = gn_stats_ref(x, eps)
    return {k: max(stats_errors(stats_as_mr(m, r), mean, rstd).values())
            for k, (m, r) in gn_stats_defects(x, eps, slots).items()}


def gn_output_sensitivity(x, gamma, beta, eps, silu, slots):
    """{defect: worst_group error of its output}."""
    y = gn_ref(x, None, gamma, beta, eps, silu)[0]
    return {k: worst_group(v, y) for k, v in gn_defect_outputs(x, gamma, beta, eps, silu, slots).items()}


def gn_bwd_sensitivity(x, mean, rstd, gamma, beta, silu, dy, chunks):
    """{defect: worst_group error of dx}: the last non-empty chunk left out of the two group sums, the last channel of
    each group (but the last) using the next group's statistics and sums, sample b using sample b+1's statistics."""
    B, HW, C = x.shape
    cpg = C // GROUPS
    dx = gn_bwd_ref(x, mean, rstd, gamma, beta, silu, dy)
    out = {}
    bounds = [b for b in slot_bounds(HW, chunks) if b[1] > b[0]]
    if len(bounds) > 1:
        out["drop_chunk"] = worst_group(gn_bwd_ref(x, mean, rstd, gamma, beta, silu, dy,
                                                   drop_rows=slice(*bounds[-1])), dx)
    if B > 1:
        out["next_sample"] = worst_group(gn_bwd_ref(x, mean.roll(-1, 0), rstd.roll(-1, 0), gamma, beta, silu, dy), dx)
    # neighbour: group g+1's sums are those of its own channels; only the moved channel's dx changes
    xd, dyd, g, b = x.double(), dy.double(), gamma.double(), beta.double()
    xh = (xd - _per_channel(mean.double(), cpg)) * _per_channel(rstd.double(), cpg)
    d = (dyd * _silu_grad(xh * g + b) if silu else dyd) * g
    m1 = d.reshape(B, HW, GROUPS, cpg).sum(dim=(1, 3)) / (HW * cpg)
    m2 = (d * xh).reshape(B, HW, GROUPS, cpg).sum(dim=(1, 3)) / (HW * cpg)
    last = torch.arange(cpg - 1, C - cpg, cpg)
    gn = (last + cpg) // cpg
    mn, rn = mean.double()[:, gn][:, None], rstd.double()[:, gn][:, None]
    xhl = (xd[..., last] - mn) * rn
    dl = (dyd[..., last] * _silu_grad(xhl * g[last] + b[last]) if silu else dyd[..., last]) * g[last]
    dxn = dx.clone()
    dxn[..., last] = rn * (dl - m1[:, gn][:, None] - xhl * m2[:, gn][:, None])
    out["neighbour"] = worst_group(dxn, dx)
    return out


def ln_sensitivity(x, gamma, beta, eps):
    """{defect: worst_row error of the LayerNorm output}: the last float4 (4 channels) left out of the row statistics,
    and row r normalised with row r+1's statistics (only with more than one row)."""
    y, mean, rstd = ln_ref(x, gamma, beta, eps)
    xd = x.double()
    out = {}
    if x.shape[-1] > 4:
        _, m, r = ln_ref(xd[..., :-4], gamma[:-4], beta[:-4], eps)
        out["drop_vec"] = worst_row((xd - m[..., None]) * r[..., None] * gamma.double() + beta.double(), y)
    if x.shape[0] > 1:
        out["next_row"] = worst_row((xd - mean.roll(-1)[..., None]) * rstd.roll(-1)[..., None] * gamma.double()
                                    + beta.double(), y)
    return out


def ln_bwd_sensitivity(x, gamma, eps, dy):
    """{defect: worst_row error of dx}: the last float4 left out of the two row sums, row r using row r+1's stats."""
    xd, dyd, g = x.double(), dy.double(), gamma.double()
    dx = ln_bwd_ref(x, gamma, eps, dy)[0]
    _, mean, rstd = ln_ref(xd, torch.ones_like(g), torch.zeros_like(g), eps)
    out = {}

    def dx_with(mean, rstd, keep):
        xh = (xd - mean[..., None]) * rstd[..., None]
        d = dyd * g
        C = x.shape[-1]
        s1 = (d[..., :keep]).sum(-1, keepdim=True) / C
        s2 = (d * xh)[..., :keep].sum(-1, keepdim=True) / C
        return rstd[..., None] * (d - s1 - xh * s2)

    if x.shape[-1] > 4:
        out["drop_vec"] = worst_row(dx_with(mean, rstd, x.shape[-1] - 4), dx)
    if x.shape[0] > 1:
        out["next_row"] = worst_row(dx_with(mean.roll(-1), rstd.roll(-1), x.shape[-1]), dx)
    return out
