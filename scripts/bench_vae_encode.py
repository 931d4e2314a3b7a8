"""VAE encoder throughput: encode B x 512^2 images (AutoencoderKL(with_encoder=True), synthetic weights), and the
asymmetric-pad stride-2 conv (af_conv3x3_down01_bf16) against the pad-1 stride-2 conv (af_conv3x3_bf16) at the
encoder's three Downsample shapes, alternated in one process.  Prints the card and its power limit with the numbers.

    python scripts/bench_vae_encode.py [--batch 8] [--reps 10]
"""
import argparse
import subprocess
import sys

import torch

sys.path.insert(0, ".")


def encoder_flops(B, H, W, ch=128, ch_mult=(1, 2, 4, 4), num_res_blocks=2, z_channels=4):
    """Multiply-adds x 2 of every conv / GEMM of the encoder (plus the folded quant_conv), counted from the layer shapes.
    GroupNorm, SiLU and softmax are not counted."""
    conv = lambda h, w, ci, co, k: 2.0 * h * w * ci * co * k * k
    f = conv(H, W, 3, ch, 3)
    h, w, cin = H, W, ch
    for i, m in enumerate(ch_mult):
        cout = ch * m
        for _ in range(num_res_blocks):
            f += conv(h, w, cin, cout, 3) + conv(h, w, cout, cout, 3) + (conv(h, w, cin, cout, 1) if cin != cout else 0)
            cin = cout
        if i != len(ch_mult) - 1:
            h, w = h // 2, w // 2
            f += conv(h, w, cin, cin, 3)
    for _ in range(2):                                                 # mid.block_1 / block_2
        f += 2 * conv(h, w, cin, cin, 3)
    n = h * w
    f += 4 * conv(h, w, cin, cin, 1) + 2 * 2.0 * n * n * cin           # q, k, v, proj_out; scores and P.V
    f += conv(h, w, cin, 2 * z_channels, 3)
    return B * f


def time_ms(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_vae_encode: no CUDA device")
    from adaprompt_b200 import ops
    from adaprompt_b200.packing import pack_conv3x3
    from adaprompt_b200.vae import AutoencoderKL, encode_first_stage
    from adaprompt_b200.weights import spec_of, synth_state_dict

    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    print(f"device: {card[0] if card else torch.cuda.get_device_name()}")

    with torch.device("meta"):
        vae = AutoencoderKL(with_encoder=True)
    vae = vae.to_empty(device="cuda")
    vae.load_state_dict(synth_state_dict(spec_of(vae), 1235))
    vae.eval()
    B = args.batch
    x = (torch.rand(B, 3, 512, 512, generator=torch.Generator().manual_seed(0)) * 2 - 1).cuda()
    for _ in range(2):
        encode_first_stage(vae, x)
    ms = time_ms(lambda: encode_first_stage(vae, x), args.reps)
    fl = encoder_flops(B, 512, 512)
    print(f"encode {B} x 512^2: {ms:.2f} ms, {B / ms * 1e3:.2f} images/s, {fl / ms / 1e9:.1f} TFLOP/s algorithmic "
          f"({fl / B / 1e12:.3f} TFLOP per image, counted from the layer shapes)")

    print("stride-2 conv at the encoder's Downsample shapes (us per launch, alternated, L2 not flushed):")
    for C, H in ((128, 512), (256, 256), (512, 128)):
        xb = torch.randn(B, H, H, C, device="cuda").bfloat16()
        wp = pack_conv3x3((torch.randn(C, C, 3, 3, device="cuda") * 0.02).bfloat16())
        bias = torch.zeros(C, device="cuda")
        out = torch.empty(B, H // 2, H // 2, C, device="cuda")
        st = ops.gn_stats_for_conv(B, H // 2, H // 2, C, "cuda")
        down01 = lambda: ops.conv3x3_down01(xb, wp, out, bias=bias, gn_stats=st.buf)
        pad1 = lambda: ops.conv3x3(xb, wp, out, stride=2, bias=bias, gn_stats=st.buf)
        for f in (down01, pad1):
            time_ms(f, 3)
        a, b = [], []
        for _ in range(5):
            a.append(time_ms(down01, 20))
            b.append(time_ms(pad1, 20))
        a_ms, b_ms = min(a), min(b)
        print(f"  B{B} C{C} {H}x{H} -> {H // 2}x{H // 2}: down01 {a_ms * 1e3:.1f} us, pad-1 {b_ms * 1e3:.1f} us, "
              f"ratio {a_ms / b_ms:.3f}")


if __name__ == "__main__":
    main()
