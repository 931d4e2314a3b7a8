"""CPU checks of the first-stage encoder and img2img host logic: state_dict layout of AutoencoderKL(with_encoder=True),
argument checks of the new entry points (no GPU needed), and the t_enc range check that runs before any device work."""
import pytest
import torch


def test_autoencoder_with_encoder_has_reference_state_dict_keys():
    from adaprompt_b200.vae import AutoencoderKL
    from oracle.vae_oracle import VAESpec
    from vae_encoder_oracle import full_state_spec
    with torch.device("meta"):
        vae = AutoencoderKL(with_encoder=True)
    spec = full_state_spec(VAESpec())
    mine = [(k, tuple(v.shape)) for k, v in vae.state_dict().items()]
    assert mine == list(spec.items())
    full = {k: torch.empty(s, device="meta") for k, s in spec.items()}
    full["loss.logvar"] = torch.empty((), device="meta")
    full["loss.discriminator.main.0.weight"] = torch.empty(64, 3, 4, 4, device="meta")
    vae.load_state_dict(full, assign=True)                       # strict: encoder and quant_conv kept, loss.* dropped
    with pytest.raises(RuntimeError):                            # a missing encoder key still fails the strict load
        vae.load_state_dict({k: v for k, v in full.items() if k != "encoder.conv_in.weight"}, assign=True)


def test_default_autoencoder_is_unchanged_and_encode_needs_the_encoder():
    from adaprompt_b200.vae import AutoencoderKL
    from oracle.vae_oracle import VAESpec
    with torch.device("meta"):
        vae = AutoencoderKL()
    assert list(vae.state_dict()) == list(VAESpec().state_spec())
    with pytest.raises(NotImplementedError):
        vae.encode(torch.zeros(1, 3, 64, 64))


def test_encode_has_no_cpu_fallback_and_rejects_the_mask():
    from adaprompt_b200.vae import AutoencoderKL, Downsample
    vae = AutoencoderKL(ddconfig=dict(double_z=True, z_channels=4, resolution=64, in_channels=3, out_ch=3, ch=64,
                                      ch_mult=[1, 1], num_res_blocks=1, attn_resolutions=[], dropout=0.0),
                        with_encoder=True)
    with pytest.raises(RuntimeError):
        vae.encode(torch.zeros(1, 3, 64, 64))
    with pytest.raises(NotImplementedError):
        vae.encode(torch.zeros(1, 3, 64, 64), mask=torch.ones(1, 1, 64, 64))
    with pytest.raises(NotImplementedError):
        Downsample(64, with_conv=False)


def test_new_entry_points_reject_bad_arguments_without_a_gpu(lib):
    from ctypes import byref
    from adaprompt_b200._lib import AfEpilogue
    ep = AfEpilogue()
    ep.out = 16
    down = lambda C, H, W, Cout: lib.af_conv3x3_down01_bf16(16, C, 16, 1, H, W, Cout, byref(ep), 0, None)
    assert down(64, 9, 8, 64) < 0 and b"even" in lib.af_last_error()            # odd H
    assert down(64, 8, 7, 64) < 0 and b"even" in lib.af_last_error()            # odd W
    assert down(96, 8, 8, 64) < 0 and b"multiple of 64" in lib.af_last_error()  # C % 64
    assert down(64, 8, 8, 12) < 0 and b"multiple of 8" in lib.af_last_error()   # Cout % 8
    assert lib.af_conv3x3_down01_bf16(None, 64, 16, 1, 8, 8, 64, byref(ep), 0, None) < 0
    assert lib.af_conv_in(16, 16, None, 16, 1, 5, 8, 8, 128, None) < 0 and b"Cin=5" in lib.af_last_error()
    assert lib.af_vae_posterior(16, 1, 64, 0, None, 1.0, 16, None, None, None) < 0 and b"zc=0" in lib.af_last_error()
    assert lib.af_vae_posterior(None, 1, 64, 4, None, 1.0, 16, None, None, None) < 0


@pytest.mark.parametrize("strength,steps,t_enc", [(0.75, 4, 3), (0.5, 50, 25), (0.04, 50, 2), (0.98, 50, 49),
                                                  (0.8, 5, 4)])
def test_img2img_t_enc_accepts_the_valid_range(strength, steps, t_enc):
    from adaprompt_b200.ddim import img2img_t_enc
    assert img2img_t_enc(strength, steps) == t_enc


@pytest.mark.parametrize("strength,steps", [(1.0, 50), (1.0, 4), (0.03, 50), (0.0, 50), (0.5, 2), (0.3, 4), (-0.5, 50)])
def test_img2img_t_enc_rejects_what_the_device_cannot_run(strength, steps):
    from adaprompt_b200.ddim import img2img_t_enc
    with pytest.raises(ValueError, match="t_enc"):
        img2img_t_enc(strength, steps)


def test_cli_rejects_a_bad_strength_before_building_anything(capsys):
    from adaprompt_b200 import txt2img
    with pytest.raises(SystemExit):
        txt2img.parse_args(["--synthetic", "--init_img", "x.png", "--strength", "1.0", "--ddim_steps", "4"])
    assert "t_enc" in capsys.readouterr().err
    args = txt2img.parse_args(["--synthetic", "--init_img", "x.png", "--ddim_steps", "4"])
    assert args.strength == 0.75
    assert txt2img.parse_args(["--synthetic", "--strength", "1.0"]).init_img is None   # txt2img ignores --strength
