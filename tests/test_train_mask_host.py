"""CPU checks of the masked Stage-1 step (image-masked batches): the masked reconstruction loss against a float64
restatement, the host-side rejection of malformed masks before any device work, and the new C-ABI symbols in the
header and the binding table."""
import os
import re

import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _recon_loss64(eps, target, img, fg, fgw, bgw):
    """calc_recon_loss (ddpm.py:3571-3595) as the issue restates it, in float64 with explicit channel broadcast."""
    e, t = eps.double(), target.double()
    C = e.shape[1]
    img = torch.ones_like(e[:, :1]) if img is None else img.double()
    fg = torch.ones_like(e[:, :1]) if fg is None else fg.double()
    img, fg = img.expand(-1, C, -1, -1), fg.expand(-1, C, -1, -1)
    pix = (e * img - t * img) ** 2
    wf, wb = fg * img * fgw, (1 - fg) * img * bgw
    return ((pix * wf).sum() + (pix * wb).sum()) / (wf.sum() + wb.sum())


def _masks(B, H, seed):
    from adaprompt_b200.synthetic import synthetic_masks
    return synthetic_masks(B, H, torch.Generator().manual_seed(seed))


@pytest.mark.parametrize("which", ["both", "img", "fg", "bool"])
@pytest.mark.parametrize("fgw,bgw", [(1.0, 1.0), (4.0, 0.25), (0.5, 3.0)])
def test_calc_recon_loss_matches_float64_restatement(which, fgw, bgw):
    from adaprompt_b200.train import calc_recon_loss
    g = torch.Generator().manual_seed(3)
    B, H = 3, 16
    eps, target = torch.randn(B, 4, H, H, generator=g), torch.randn(B, 4, H, H, generator=g)
    img, fg = _masks(B, H, 7)
    if which == "img":
        fg = None
    elif which == "fg":
        img = None
    elif which == "bool":
        img, fg = img.bool(), fg.bool()
    got = calc_recon_loss(eps, target, img, fg, fgw, bgw)
    want = _recon_loss64(eps, target, img, fg, fgw, bgw)
    assert abs(got.double().item() - want.item()) < 1e-6 * want.item(), (got.item(), want.item())


def test_calc_recon_loss_without_masks_is_mse():
    from adaprompt_b200.train import calc_recon_loss
    g = torch.Generator().manual_seed(4)
    eps, target = torch.randn(2, 4, 8, 8, generator=g), torch.randn(2, 4, 8, 8, generator=g)
    for w in ((1.0, 1.0), (3.0, 0.5)):
        got, want = calc_recon_loss(eps, target, None, None, *w), F.mse_loss(eps, target)
        assert abs(got.item() - want.item()) < 1e-6 * want.item()


def test_calc_recon_loss_ignores_pixels_outside_the_image():
    """Whatever eps / target hold where img_mask is 0 (here 1e6) does not change the loss."""
    from adaprompt_b200.train import calc_recon_loss
    g = torch.Generator().manual_seed(5)
    eps, target = torch.randn(2, 4, 16, 16, generator=g), torch.randn(2, 4, 16, 16, generator=g)
    img, fg = _masks(2, 16, 1)
    base = calc_recon_loss(eps, target, img, fg, 2.0, 0.5)
    dirty = eps + (1 - img) * 1e6
    assert torch.equal(calc_recon_loss(dirty, target, img, fg, 2.0, 0.5), base)


def test_synthetic_masks_are_opt_in_and_plausible():
    from adaprompt_b200.synthetic import stage1_batch
    plain = stage1_batch("cpu", 4, 32, torch.Generator().manual_seed(2))
    masked = stage1_batch("cpu", 4, 32, torch.Generator().manual_seed(2), masks=True)
    assert set(masked) - set(plain) == {"img_mask", "fg_mask"}
    assert all(torch.equal(plain[k], masked[k]) for k in plain)
    img, fg = masked["img_mask"], masked["fg_mask"]
    assert img.shape == fg.shape == (4, 1, 32, 32)
    assert ((fg == 0) | (img == 1)).all(), "the face lies inside the image"
    frac = img.mean((1, 2, 3))
    assert (frac > 0.5).all() and (fg.sum((1, 2, 3)) > 0).all()


def _batch(B=2, H=8):
    g = torch.Generator().manual_seed(0)
    return {"x0": torch.randn(B, 4, H, H, generator=g), "t": torch.zeros(B, dtype=torch.long)}


@pytest.mark.parametrize("bad,match", [
    (lambda b: torch.ones(2, 8, 8), "shape"),                           # no channel dim
    (lambda b: torch.ones(2, 1, 4, 4), "shape"),                        # not at latent resolution
    (lambda b: torch.ones(3, 1, 8, 8), "shape"),                        # batch mismatch
    (lambda b: torch.ones(2, 4, 8, 8), "shape"),                        # one mask per channel
    (lambda b: torch.ones(2, 1, 8, 8, dtype=torch.int32), "float or bool"),
    (lambda b: [[1.0]], "tensor"),
], ids=["3d", "lowres", "batch", "channels", "int", "list"])
def test_bad_masks_raise_before_device_work(bad, match):
    from adaprompt_b200.train_cond import batch_masks
    for key in ("img_mask", "fg_mask"):
        b = _batch()
        b[key] = bad(b)
        with pytest.raises(ValueError, match=match):
            batch_masks(b)


def test_unet_forward_train_rejects_bad_img_mask_before_device_work():
    from adaprompt_b200.train import unet_forward_train
    x = torch.zeros(2, 4, 8, 8)
    extra = {"use_layerwise_context": True, "img_mask": torch.ones(2, 1, 16, 16)}
    with pytest.raises(ValueError, match="img_mask"):
        unet_forward_train(None, x, torch.zeros(2), torch.zeros(32, 77, 768), extra)
    with pytest.raises(NotImplementedError):
        unet_forward_train(None, x, torch.zeros(2), torch.zeros(32, 77, 768),
                           {"use_layerwise_context": True, "capture_distill_attn": True})


def test_micro_batches_must_agree_on_their_masks():
    from adaprompt_b200.train_cond import check_mask_presence
    m = torch.ones(2, 1, 8, 8)
    check_mask_presence([_batch(), _batch()])
    check_mask_presence([dict(_batch(), img_mask=m, fg_mask=m), dict(_batch(), img_mask=m, fg_mask=m)])
    for other in (dict(_batch(), img_mask=m), dict(_batch(), fg_mask=m), _batch()):
        with pytest.raises(ValueError, match="disagree"):
            check_mask_presence([dict(_batch(), img_mask=m, fg_mask=m), other])


def test_key_mask_argument_checks():
    """ops.check_key_mask (ops.attention_bwd / ops.bgemm with key_mask, AttentionFn): uint8 [B, N], contiguous, CUDA."""
    from adaprompt_b200 import ops
    with pytest.raises(ValueError, match="uint8"):
        ops.check_key_mask(torch.ones(2, 128, dtype=torch.bool), 2, 128)
    with pytest.raises(ValueError, match="shape"):
        ops.check_key_mask(torch.ones(2, 64, dtype=torch.uint8), 2, 128)
    with pytest.raises(ValueError, match="shape"):
        ops.check_key_mask(torch.ones(1, 2, 128, dtype=torch.uint8), 2, 128)
    with pytest.raises(ValueError, match="contiguous"):
        ops.check_key_mask(torch.ones(128, 2, dtype=torch.uint8).t(), 2, 128)
    with pytest.raises(ValueError, match="CUDA"):
        ops.check_key_mask(torch.ones(2, 128, dtype=torch.uint8), 2, 128)
    with pytest.raises(ValueError, match="Tensor"):
        ops.check_key_mask(None, 2, 128)
    z = torch.zeros(256, 8)
    with pytest.raises(ValueError, match="uint8"):        # rejected before the library is touched
        ops.attention_bwd(z, z, z, z, z, z, z, z, z, B=2, heads=8, N=128, d=40,
                          key_mask=torch.ones(2, 128, dtype=torch.float32))
    with pytest.raises(ValueError, match="mode 0"):
        ops.bgemm(z, 8, (0, 0), z, 8, (0, 0), z, 8, (0, 0), M=8, N=8, K=8, nb0=1, nb1=1, mode=0,
                  key_mask=torch.ones(1, 8, dtype=torch.uint8))


def test_masked_entry_points_are_declared_and_bound(lib):
    from adaprompt_b200 import _lib
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "adaface_b200.h")).read(), flags=re.S)
    for name in ("af_attention_bwd_masked_bf16", "af_bgemm_masked_bf16"):
        assert re.search(rf"\b{name}\s*\(", src), name
        assert name in _lib.SIGNATURES and hasattr(lib._cdll, name), name
    assert lib.af_version() == 202


def test_masked_entry_points_reject_bad_arguments_without_a_gpu(lib):
    from ctypes import byref
    from adaprompt_b200._lib import AfBgemm
    args = [1, 48, 1, 48, 1, 48, 1, 48, 1, 256, 1, 256, 1, 256, 1, 1]
    rc = lib.af_attention_bwd_masked_bf16(*args, None, 1, 48, 1, 48, 1, 40, 2, 1, 128, 40, None)
    assert rc < 0 and b"key_mask" in lib.af_last_error()
    rc = lib.af_attention_bwd_masked_bf16(*args, 16, 1, 48, 1, 48, 1, 40, 2, 1, 192, 40, None)
    assert rc < 0 and b"multiple of 128" in lib.af_last_error()
    g = AfBgemm()
    g.A, g.B, g.C, g.vec = 16, 16, 16, 16
    g.lda = g.ldb = g.ldc = 8
    g.M = g.N = g.K = 8
    g.nb0 = g.nb1 = 1
    g.mode = 1
    assert lib.af_bgemm_masked_bf16(byref(g), None, 8, 0, None) < 0 and b"null key_mask" in lib.af_last_error()
    g.mode = 0
    assert lib.af_bgemm_masked_bf16(byref(g), 16, 8, 0, None) < 0 and b"mode 0" in lib.af_last_error()
