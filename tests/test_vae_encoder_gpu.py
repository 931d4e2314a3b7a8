"""B200 checks of the first-stage encoder (adaprompt_b200/vae.py -> C ABI -> sm_100a kernels) and the img2img path.

Kernels against float64 / torch references on the same operands; the encoder against the fp32 oracle of
tests/vae_encoder_oracle.py; the CLI img2img run against the
oracle chain encoder -> posterior -> stochastic_encode -> DDIM decode on the UNet oracle -> decoder.

Limits are about twice the worst value measured on one B200 (1000 W power limit): down01 rel-L2 3.3e-6, worst pixel
4.1e-6, last row / column 1.9e-6; conv_in 1.2e-7; encoder posterior mean / logvar 8.7e-3 (the decoder's end-of-pipeline
budget is 2e-2); sampler steps 1.5e-7; CLI img2img z_enc 1.3e-4, latents 4.4e-3, PNG 0.34 grey levels."""
import os

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
ENC_TOL = 1.75e-2


def _rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return ((a - b).norm() / b.norm()).item()


def _bf16(t):
    return t.to(torch.bfloat16)


# ------------------------------------------------------------------------------------------ stride-2 conv, pad (0,1,0,1)
def _down_case(B, C, H, W, Cout, seed, x=None):
    from adaprompt_b200.packing import pack_conv3x3
    g = torch.Generator().manual_seed(seed)
    x = _bf16(torch.randn(B, H, W, C, generator=g)) if x is None else x
    w = _bf16(torch.randn(Cout, C, 3, 3, generator=g) / (3 * C ** 0.5))
    b = torch.randn(Cout, generator=g)
    return x, w, b, pack_conv3x3(w.float().cuda())


def _down_ref(x, w, b):
    xd = x.cuda().double().permute(0, 3, 1, 2)
    y = F.conv2d(F.pad(xd, (0, 1, 0, 1)), w.cuda().double(), b.cuda().double(), stride=2)
    return y.permute(0, 2, 3, 1)


def _down_run(x, wp, b, Cout, **kw):
    from adaprompt_b200 import ops
    B, H, W, _ = x.shape
    out = torch.empty(B, H // 2, W // 2, Cout, dtype=torch.float32, device="cuda")
    ops.conv3x3_down01(x.cuda(), wp, out, bias=b.cuda(), **kw)
    return out


def _down_check(out, ref, what):
    """global rel-L2, worst output pixel (its channel vector against the RMS pixel norm), and the last output row and
    column (the taps that read the pad) on their own."""
    d = (out.double() - ref)
    rms = ref.norm(dim=-1).pow(2).mean().sqrt()
    glob = (d.norm() / ref.norm()).item()
    worst = (d.norm(dim=-1) / rms).max().item()
    edge = max((d[:, -1].norm() / ref[:, -1].norm()).item(), (d[:, :, -1].norm() / ref[:, :, -1].norm()).item())
    print(f"down01 {what}: rel-L2 {glob:.2e}, worst pixel {worst:.2e}, last row/col {edge:.2e}")
    assert glob < 7e-6 and worst < 9e-6 and edge < 4e-6, what


ENCODER_SHAPES = [(1, 128, 512), (8, 128, 512), (1, 256, 256), (8, 256, 256), (1, 512, 128), (8, 512, 128)]
SMALL_SHAPES = [(3, 64, 10, 14, 72), (2, 192, 6, 34, 136), (1, 64, 2, 2, 8), (5, 128, 24, 40, 256)]


@pytest.mark.parametrize("B,C,H", ENCODER_SHAPES)
def test_conv3x3_down01_encoder_shapes_match_float64(B, C, H):
    x, w, b, wp = _down_case(B, C, H, H, C, seed=B * 7 + C)
    out = _down_run(x, wp, b, C)
    _down_check(out, _down_ref(x, w, b), f"B{B} C{C} {H}x{H}")


@pytest.mark.parametrize("B,C,H,W,Cout", SMALL_SHAPES)
def test_conv3x3_down01_odd_tiles_match_float64(B, C, H, W, Cout):
    x, w, b, wp = _down_case(B, C, H, W, Cout, seed=H * W + C)
    out = _down_run(x, wp, b, Cout)
    _down_check(out, _down_ref(x, w, b), f"B{B} C{C} {H}x{W} -> {Cout}")


@pytest.mark.parametrize("B,C,H,W,Cout", [(1, 128, 512, 512, 128), (8, 512, 128, 128, 512), (5, 128, 24, 40, 256)])
def test_conv3x3_down01_schedules_agree(B, C, H, W, Cout):
    """CTA pairs or not: bit-identical (same accumulation order); split-K: same values to fp32 rounding."""
    from adaprompt_b200 import ops
    x, w, b, wp = _down_case(B, C, H, W, Cout, seed=3)
    with ops.launch_options(pair_mode=1, split_k=1):
        never = _down_run(x, wp, b, Cout)
    with ops.launch_options(pair_mode=2, split_k=1):
        always = _down_run(x, wp, b, Cout)
    with ops.launch_options(pair_mode=1, split_k=0):
        split = _down_run(x, wp, b, Cout)
    assert torch.equal(never, always)
    assert _rel(split, never) < 1e-6
    _down_check(split, _down_ref(x, w, b), f"split auto B{B} C{C} {H}x{W}")


def test_conv3x3_down01_reads_nothing_outside_the_image():
    """The image sits at the start of a larger buffer whose tail holds +-2^100: the bottom / right pad is TMA zero fill,
    so the result is bit-identical to the run on a buffer with nothing behind the image."""
    B, C, H, W, Cout = 2, 128, 16, 24, 128
    x, w, b, wp = _down_case(B, C, H, W, Cout, seed=11)
    big = torch.empty(B * H + 3, W, C, dtype=torch.bfloat16)
    big[:B * H] = x.reshape(B * H, W, C)
    tail = torch.full((3, W, C), 2.0 ** 100)
    tail[1::2] *= -1
    big[B * H:] = tail.to(torch.bfloat16)
    big = big.cuda()
    poisoned = _down_run(big[:B * H].view(B, H, W, C), wp, b, Cout)
    clean = _down_run(x, wp, b, Cout)
    assert torch.isfinite(poisoned).all() and torch.equal(poisoned, clean)


def test_conv3x3_down01_groupnorm_statistics():
    """gn_stats from the epilogue equal the statistics pass over the written output."""
    from adaprompt_b200 import ops
    B, C, H = 2, 256, 64
    x, w, b, wp = _down_case(B, C, H, H, C, seed=5)
    out = torch.empty(B, H // 2, H // 2, C, dtype=torch.float32, device="cuda")
    st = ops.gn_stats_for_conv(B, H // 2, H // 2, C, "cuda")
    ops.conv3x3_down01(x.cuda(), wp, out, bias=b.cuda(), gn_stats=st.buf)
    gamma, beta = torch.ones(C, device="cuda"), torch.zeros(C, device="cuda")
    y1 = torch.empty(B, H // 2, H // 2, C, dtype=torch.bfloat16, device="cuda")
    y2 = torch.empty_like(y1)
    ops.groupnorm_apply(out, st, gamma, beta, 1e-6, True, y1)
    ops.groupnorm_apply(out, ops.groupnorm_stats(out), gamma, beta, 1e-6, True, y2)
    assert _rel(y1, y2) < 1e-3


# ------------------------------------------------------------------------------------------ conv_in with 3 channels
@pytest.mark.parametrize("B,H,W", [(2, 40, 72), (1, 512, 512), (3, 64, 33)])
def test_conv_in_three_channels_matches_float64(B, H, W):
    from adaprompt_b200 import ops
    g = torch.Generator().manual_seed(H + W)
    x = torch.rand(B, 3, H, W, generator=g) * 2 - 1
    w = torch.randn(128, 3, 3, 3, generator=g) / 5
    b = torch.randn(128, generator=g)
    y = torch.empty(B, H, W, 128, dtype=torch.float32, device="cuda")
    ops.conv_in(x.cuda(), w.cuda(), b.cuda(), y)
    ref = F.conv2d(x.cuda().double(), w.cuda().double(), b.cuda().double(), padding=1).permute(0, 2, 3, 1)
    e = _rel(y, ref)
    print(f"conv_in Cin 3 B{B} {H}x{W}: rel-L2 {e:.2e}")
    assert e < 3e-7


# ------------------------------------------------------------------------------------------ posterior kernel
def test_vae_posterior_is_bit_identical_to_torch():
    from adaprompt_b200 import ops
    g = torch.Generator().manual_seed(9)
    B, H, W, zc = 3, 20, 24, 4
    m = torch.randn(B, H, W, 2 * zc, generator=g)
    m[..., zc:] = m[..., zc:] * 25 - 5                 # logvar in about [-80, 70]: both clamp bounds are exercised
    m[0, 0, 0, zc:] = torch.tensor([-30.5, 20.5, -1e4, 1e4])
    noise = torch.randn(B, zc, H, W, generator=g).cuda()
    mc = m.cuda()
    z = torch.empty(B, zc, H, W, device="cuda")
    mean, logvar = torch.empty_like(z), torch.empty_like(z)
    ops.vae_posterior(mc, noise, 0.18215, z, mean, logvar)
    params = mc.permute(0, 3, 1, 2).contiguous()
    r_mean, r_lv = torch.chunk(params, 2, dim=1)          # distributions.py:27-30, torch CUDA ops
    r_lv = torch.clamp(r_lv, -30.0, 20.0)
    r_std = torch.exp(0.5 * r_lv)
    r_z = 0.18215 * (r_mean + r_std * noise)
    assert (r_lv == -30.0).any() and (r_lv == 20.0).any()
    assert torch.equal(mean, r_mean) and torch.equal(logvar, r_lv)
    assert torch.equal(z, r_z)
    ops.vae_posterior(mc, None, 0.18215, z)                # the mode
    assert torch.equal(z, 0.18215 * r_mean)


# ------------------------------------------------------------------------------------------ encoder vs the oracle
@pytest.fixture(scope="module")
def vae_and_sd():
    from adaprompt_b200.vae import AutoencoderKL
    from adaprompt_b200.weights import synth_state_dict
    from oracle.vae_oracle import VAESpec
    from vae_encoder_oracle import full_state_spec
    sd = synth_state_dict(full_state_spec(VAESpec()), 1235)
    with torch.device("meta"):
        vae = AutoencoderKL(with_encoder=True)
    vae = vae.to_empty(device="cuda")
    vae.load_state_dict(sd)
    vae.eval()
    return vae, sd


def _check_posterior(post, ref_moments, what, limit=ENC_TOL):
    from vae_encoder_oracle import posterior
    r_mean, r_lv, _ = posterior(ref_moments)
    em, el = _rel(post.mean, r_mean), _rel(post.logvar, r_lv)
    print(f"encoder {what}: mean rel-L2 {em:.3e}, logvar rel-L2 {el:.3e}")
    assert em < limit and el < limit


@pytest.mark.parametrize("B,H", [(2, 64), (1, 128), (1, 256)])
def test_encoder_matches_the_cpu_oracle(vae_and_sd, B, H):
    from oracle.vae_oracle import VAESpec
    from vae_encoder_oracle import encode, seeded_images
    vae, sd = vae_and_sd
    x = seeded_images(B, H, H, seed=H + B)
    post = vae.encode(x.cuda())
    torch.cuda.synchronize()
    assert post.mean.shape == (B, 4, H // 8, H // 8)
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    with torch.no_grad():
        ref = encode(sd, VAESpec(), x)
    _check_posterior(post, ref, f"B{B} {H}x{H}")


def test_encoder_512px_matches_the_oracle_on_the_gpu(vae_and_sd):
    from oracle.vae_oracle import VAESpec
    from vae_encoder_oracle import encode, seeded_images
    vae, sd = vae_and_sd
    x = seeded_images(2, 512, 512, seed=512).cuda()
    post = vae.encode(x)
    prev = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.no_grad():
            ref = encode({k: v.cuda() for k, v in sd.items()}, VAESpec(), x)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev
    _check_posterior(post, ref, "B2 512x512 (oracle on the GPU, fp32, TF32 off)")
    again = vae.encode(x)
    assert torch.equal(post.mean, again.mean) and torch.equal(post.logvar, again.logvar)     # run to run


def test_encode_first_stage_chunking_is_bit_identical(vae_and_sd):
    from adaprompt_b200 import ops
    from adaprompt_b200.vae import encode_first_stage
    from vae_encoder_oracle import seeded_images
    vae, _ = vae_and_sd
    x = seeded_images(3, 128, 128, seed=3).cuda()
    with ops.launch_options(split_k=1):        # whole-tile GEMM schedule: a sample's arithmetic is independent of the batch
        whole = encode_first_stage(vae, x)
        chunked = encode_first_stage(vae, x, max_batch=1)
    assert torch.equal(whole.mean, chunked.mean) and torch.equal(whole.logvar, chunked.logvar)
    assert torch.equal(whole.parameters[:, :4], whole.mean)                    # NCHW (mean | raw logvar)


def test_first_stage_encoding_draws_the_reference_noise(vae_and_sd):
    """get_first_stage_encoding(encode_first_stage(x)) under torch.manual_seed(s) equals
    scale * (mean + std * torch.randn(mean.shape)) drawn under the same seed: the global CPU RNG is used as upstream."""
    from adaprompt_b200.ldm_lite import LatentDiffusionLite
    from vae_encoder_oracle import seeded_images
    vae, _ = vae_and_sd
    ldm = LatentDiffusionLite(unet=torch.nn.Identity(), first_stage_model=vae).cuda()
    x = seeded_images(2, 64, 64, seed=8).cuda()
    torch.manual_seed(1234)
    post = ldm.encode_first_stage(x)
    z = ldm.get_first_stage_encoding(post)
    after = torch.randn(1)
    torch.manual_seed(1234)
    noise = torch.randn(post.mean.shape)
    assert torch.equal(torch.randn(1), after)                                  # the stream advanced by one draw
    ref = ldm.scale_factor * (post.mean + post.std * noise.cuda())
    assert torch.equal(z, ref)
    assert torch.equal(ldm.get_first_stage_encoding(post.mean), ldm.scale_factor * post.mean)
    assert torch.equal(post.mode(), post.mean) and torch.equal(post.var, torch.exp(post.logvar))


# ------------------------------------------------------------------------------------------ sampler steps
def test_stochastic_encode_and_decode_match_the_oracle():
    from adaprompt_b200.ddim import DDIMSampler
    from adaprompt_b200.ldm_lite import LatentDiffusionLite
    from vae_encoder_oracle import ddim_decode, stochastic_encode
    S, t_enc, b = 10, 7, 2
    g = torch.Generator().manual_seed(17)
    x0, noise = torch.randn(b, 4, 16, 16, generator=g), torch.randn(b, 4, 16, 16, generator=g)
    cc, cu = torch.randn(b, 4, 16, 16, generator=g), torch.randn(b, 4, 16, 16, generator=g)

    def apply(x, t, c):          # a smooth stand-in for the UNet: depends on x, t and the conditioning
        return 0.3 * x + c[0] * (t.float() / 1000.0).view(-1, 1, 1, 1).to(x.device)

    ldm = LatentDiffusionLite(unet=torch.nn.Identity()).cuda()
    ldm.apply_model = apply
    sampler = DDIMSampler(ldm)
    sampler.make_schedule(ddim_num_steps=S, ddim_eta=0.0, verbose=False)
    z = sampler.stochastic_encode(x0.cuda(), torch.full((b,), t_enc, dtype=torch.long, device="cuda"), noise=noise.cuda())
    ref_z = stochastic_encode(x0, t_enc, S, noise)
    assert _rel(z, ref_z) < 1e-6
    cond, uncond = (cc.cuda(), ["p"] * b, {}), (cu.cuda(), [""] * b, {})
    out = sampler.decode(z, cond, t_enc, guidance_scale=7.5, unconditional_conditioning=uncond)
    ref = ddim_decode(apply, S, ref_z, (cc, ["p"] * b, {}), (cu, [""] * b, {}), t_enc, 7.5)
    e = _rel(out, ref)
    print(f"stochastic_encode + decode vs oracle: rel-L2 {e:.2e}")
    assert e < 3e-7


# ------------------------------------------------------------------------------------------ CLI and wrapper
def _write_init_png(path, H, W):
    import numpy as np
    from PIL import Image
    from vae_encoder_oracle import seeded_images
    x = seeded_images(1, H, W, seed=42)[0]
    Image.fromarray((255. * (x + 1) / 2).permute(1, 2, 0).numpy().round().clip(0, 255).astype(np.uint8)).save(path)


def test_img2img_cli_matches_the_oracle_pipeline(tmp_path):
    """CLI img2img at 256^2, 4 steps, strength 0.75 (t_enc 3) against the oracle chain fed the noises the CLI saved:
    encoder -> posterior -> scale -> stochastic_encode -> DDIM decode on the UNet oracle -> decoder."""
    import numpy as np
    from PIL import Image
    from adaprompt_b200 import txt2img
    from adaprompt_b200.txt2img import load_init_image
    from adaprompt_b200.weights import synth_state_dict
    from oracle.golden_inputs import EXTRA_INFO
    from oracle.unet_oracle import UNetSpec, unet_forward
    from oracle.vae_oracle import VAESpec, decode_first_stage as oracle_decode
    from vae_encoder_oracle import ddim_decode, encode, full_state_spec, posterior, stochastic_encode
    init = str(tmp_path / "init.png")
    _write_init_png(init, 256, 256)
    txt2img.main(["--synthetic", "--synthetic_clip_layers", "2", "--prompt", "a photo of a z", "--ddim_steps", "4",
                  "--n_samples", "1", "--H", "256", "--W", "256", "--scale", "4", "1", "--outdir", str(tmp_path / "out"),
                  "--init_img", init, "--strength", "0.75", "--save_latents", "--save_conditioning",
                  "--seed_weights", "1234"])
    files = sorted(os.listdir(tmp_path / "out" / "samples"))
    assert [f for f in files if f.endswith(".png")] == ["r0-00000.png"]
    assert Image.open(str(tmp_path / "out" / "samples" / "r0-00000.png")).size == (256, 256)
    lat = torch.load(str(tmp_path / "out" / "samples" / "r0-00000-latents.pt"))
    cond = torch.load(str(tmp_path / "out" / "samples" / "r0-00000-cond.pt"))
    assert cond["t_enc"] == 3
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    uspec, vspec = UNetSpec(), VAESpec()
    sd_u = synth_state_dict(uspec.state_spec(), 1234)
    sd_v = synth_state_dict(full_state_spec(vspec), 1235)
    apply = lambda x, t, c: unet_forward(sd_u, uspec, x, t, c[0], dict(c[2]))
    with torch.no_grad():
        mean, _, std = posterior(encode(sd_v, vspec, load_init_image(init, 256, 256)))
        init_latent = 0.18215 * (mean + std * cond["posterior_noise"])
        z_enc = stochastic_encode(init_latent, 3, 4, cond["stochastic_encode_noise"])
        ref_lat = ddim_decode(apply, 4, z_enc, (cond["c"], ["p"], dict(EXTRA_INFO)), (cond["uc"], [""], dict(EXTRA_INFO)),
                              3, 4.0)
        ref_img = torch.clamp((oracle_decode(sd_v, vspec, ref_lat) + 1.0) / 2.0, 0.0, 1.0)
    ez, e = _rel(cond["z_enc"], z_enc), _rel(lat, ref_lat)
    png = np.asarray(Image.open(str(tmp_path / "out" / "samples" / "r0-00000.png"))).astype(np.float32)
    ref_png = (255.0 * ref_img[0].permute(1, 2, 0).numpy()).round().clip(0, 255)
    mad = float(np.abs(png - ref_png).mean())
    print(f"img2img vs oracle pipeline: z_enc rel-L2 {ez:.3e}, latent rel-L2 {e:.3e}, PNG mean abs diff {mad:.2f} / 255")
    assert ez < 3e-4 and e < 1e-2 and mad < 2.0


def test_wrapper_img2img_from_an_image_and_from_latents():
    import types
    from adaprompt_b200.adaface_wrapper import AdaFaceWrapper
    from adaprompt_b200.clip_text import CLIPTextConfigLite, CLIPTextModelWrapper
    from adaprompt_b200.ldm_lite import SD15_UNET_CONFIG
    from adaprompt_b200.subj_basis_generator import SubjBasisGenerator
    from adaprompt_b200.unet import UNetModel
    from adaprompt_b200.vae import AutoencoderKL
    from adaprompt_b200.weights import spec_of, synth_state_dict
    from vae_encoder_oracle import seeded_images

    class Tok:
        pad_token_id = 49407

        def encode(self, text, add_special_tokens=False):
            return [1014]

        def __call__(self, text, max_length=77, **kw):
            texts = [text] if isinstance(text, str) else list(text)
            rows = []
            for t in texts:
                ids = [49406] + [49408 + int(w[2:]) if w.startswith("z_") else 1000 + len(w) for w in t.split()][:max_length - 2] + [49407]
                rows.append(ids + [49407] * (max_length - len(ids)))
            return types.SimpleNamespace(input_ids=torch.tensor(rows))

    with torch.device("meta"):
        unet = UNetModel(**SD15_UNET_CONFIG)
        vae = AutoencoderKL(with_encoder=True)
    unet, vae = unet.to_empty(device="cuda"), vae.to_empty(device="cuda")
    unet.load_state_dict(synth_state_dict(spec_of(unet), 1234))
    vae.load_state_dict(synth_state_dict(spec_of(vae), 1235))
    unet.eval().prepare()
    cfg = CLIPTextConfigLite(num_hidden_layers=2)
    torch.manual_seed(0)
    sbg = SubjBasisGenerator(num_out_embs_per_layer=16, clip_tokenizer=Tok(), clip_config=cfg)
    w = AdaFaceWrapper("img2img", "unused", "unused", "cuda", num_inference_steps=5, unet=unet,
                       text_encoder=CLIPTextModelWrapper(cfg), tokenizer=Tok(), subj_basis_generator=sbg,
                       arc2face_text_encoder=CLIPTextModelWrapper(cfg), vae_encoder=vae)
    w.generate_adaface_embeddings(None, gen_rand_face=True)
    img = seeded_images(1, 256, 256, seed=5)
    lat = w(img, "a photo of z in a park", guidance_scale=4.0, out_image_count=2, ref_img_strength=0.6)
    assert lat.shape == (2, 4, 32, 32) and torch.isfinite(lat).all()
    lat4 = w(torch.randn(2, 4, 32, 32, generator=torch.Generator().manual_seed(1)), "a photo of z", guidance_scale=4.0,
             out_image_count=2, ref_img_strength=0.6)
    assert lat4.shape == (2, 4, 32, 32) and torch.isfinite(lat4).all()
    with pytest.raises(ValueError, match="t_enc"):
        w(img, "a photo of z", out_image_count=2, ref_img_strength=1.0)
