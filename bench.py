#!/usr/bin/env python
"""Headline benchmark: 512^2 DDIM-50 CFG AdaFace sampling, images/sec (BASELINE.json metric, configs[2]).

    python bench.py --gpus N --steps K --warmup W            # this framework (CUDA, sm_100a)
    python bench.py --impl reference --steps K --warmup W     # reference algorithm on the host CPUs (oracle port)
    python bench.py --steps K --warmup W --dump-outputs DIR   # also write the last timed step's outputs as DIR/*.npy

One "step" = one full DDIMSampler.sample() call: 50 DDIM steps x UNet on [cond ; uncond] (batch 16) for 8
images per GPU, guidance annealed (4 -> 1), eta 0, random-init SD-1.5-architecture weights, synthetic
77-token layerwise context.  `value` keeps inputs resident in HBM; `e2e` goes through the same public API
(DDIMSampler.sample) starting from pinned HOST buffers and ending with the latents back on the host.
N > 1: one process per GPU (torchrun), batch-sharded, no data-path collective (weak scaling); timing is
CUDA events, max over ranks.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DDIM_STEPS = 50
IMAGES_PER_GPU = 8
GUIDANCE = (4.0, 1.0)
LATENT = 64
VAE_GFLOP_PER_IMAGE = 2514.5    # first-stage decoder at 64x64 latents -> 512x512 (convs + the 4096-token AttnBlock)
UNET_GFLOP_PER_SAMPLE = 803.27  # SURVEY.md section 8(d): conv 443.95 + linear 233.27 + attention 126.05


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "tflops_burst": p["bf16_tflops"],
                "tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "tflops_burst": 1590.0, "tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        # median over samples taken under load (top half of the distribution is the loaded part)
        loaded = sm[len(sm) // 2:] if sm else []
        med = loaded[len(loaded) // 2] if loaded else None
        return {"sm_mhz": med, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir: str, arrays: dict):
    """--dump-outputs: writes each tensor as out_dir/<name>.npy (float64 stays float64, everything else becomes float32)
    so that two builds run with the same arguments, hence the same seeded inputs, can be compared output for output."""
    import numpy as np
    import torch
    host = {k: v.detach().to("cpu", torch.float64 if v.dtype == torch.float64 else torch.float32).numpy()
            for k, v in arrays.items()}
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"bench.py: --dump-outputs would write {total} bytes (limit {DUMP_MAX_BYTES})")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def workload_config(world: int, graph: bool = True):
    b = IMAGES_PER_GPU
    return {"workload": "ddim50_cfg_512px_batch8_per_gpu", "ddim_steps": DDIM_STEPS, "images_per_gpu": b,
            "unet_batch": 2 * b, "guidance_scale": list(GUIDANCE), "eta": 0.0, "latent": [4, LATENT, LATENT],
            "context": [16 * b, 77, 768], "parallelism": f"dp{world}",
            "weights": "random-init SD-1.5 architecture (seed 1234)",
            "l2": "activations per UNet step (>1 GB) exceed the 126 MB L2; no explicit flush", "cuda_graph": graph}


def cpu_oracle_pair_seconds(reps: int, warmup: int):
    """Times the CPU oracle (oracle/unet_oracle.py, fp32) on ONE CFG pair (UNet batch 2, 64x64 latent)."""
    import torch
    from adaprompt_b200.weights import synth_state_dict
    from oracle.golden_inputs import EXTRA_INFO
    from oracle.unet_oracle import UNetSpec, unet_forward
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    spec = UNetSpec()
    sd = synth_state_dict(spec.state_spec(), 1234)
    g = torch.Generator().manual_seed(3)
    x = torch.randn(2, 4, LATENT, LATENT, generator=g)
    t = torch.full((2,), 501, dtype=torch.long)
    ctx = torch.randn(32, 77, 768, generator=g)
    times = []
    with torch.no_grad():
        for i in range(warmup + reps):
            t0 = time.perf_counter()
            unet_forward(sd, spec, x, t, ctx, dict(EXTRA_INFO))
            if i >= warmup:
                times.append(time.perf_counter() - t0)
    times.sort()
    return times[len(times) // 2], times, cores


def run_reference(args, emit=lambda line: print(json.dumps(line))):
    """--impl reference: the reference algorithm (fp32 oracle port of UNetModel + DDIM/CFG arithmetic) on the host
    cores.  Each step is a bounded sample of the workload: one CFG-pair UNet evaluation (UNet batch 2 = one image's
    denoising step); a 512^2 DDIM-50 image costs 50 of them, so images/s = 1 / (50 * t_pair) - an EXTRAPOLATION from the
    sample, stated in the line.  One host process whatever --gpus says: the value does not scale with N."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    med, times, cores = cpu_oracle_pair_seconds(max(1, args.steps), max(0, min(args.warmup, 1)))
    value = 1.0 / (DDIM_STEPS * med)
    line = {
        "impl": "reference", "metric": "ddim50_cfg_512x512_images_per_sec", "value": value, "unit": "images/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": med * 1e3 * DDIM_STEPS * IMAGES_PER_GPU,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(1, graph=False),
        "extrapolated": True, "host_processes": 1,
        "note": "one CPU process regardless of --gpus (rank 0 only): a ratio against an N-GPU line compares N GPUs with "
                "one host process",
        "cpu_baseline": {"value": value, "unit": "images/s", "cores": cores, "kind": "port",
                         "sample": f"{len(times)} x one CFG-pair UNet forward (UNet batch 2 of the 16, 64x64 latent, fp32), "
                                   f"median {med:.2f} s; x50 DDIM steps per image (extrapolated)"},
        "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


def gpu_oracle_legs(dev, unet, sampler_call, dev_in, extra, b):
    """Parity gate + practical GPU baseline (BASELINE.md section 3), both with the fp32 oracle port of the reference
    path (oracle/unet_oracle.py: plain torch functional ops -> cuDNN / cuBLAS eager kernels) on the SAME GPU:
      parity: eps of the timed batch-16 UNet step for one conditional and one unconditional sample, and the final latent
              of image 0 of the timed 50-step run, against the oracle with TF32 off (budgets 1e-2 / 2e-2, north_star);
      gpu_eager_baseline: the oracle's UNet step at batch 16 in fp32 (torch defaults), under bf16 and fp16 autocast."""
    import torch
    from adaprompt_b200.weights import synth_state_dict
    from oracle.golden_inputs import EXTRA_INFO
    from oracle.unet_oracle import UNetSpec, ddim_sample, unet_forward
    spec = UNetSpec()
    sd = {k: v.to(dev) for k, v in synth_state_dict(spec.state_spec(), 1234).items()}
    rel = lambda a, r: float((a.float() - r.float()).norm() / r.float().norm())
    tf32 = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    x_in = torch.cat([dev_in[2]] * 2)
    t_in = torch.full((2 * b,), 501.0, device=dev)
    c2 = torch.cat([dev_in[0], dev_in[1]])
    out = {}
    with torch.no_grad():
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = False
        eps = unet(x_in, t_in, context=c2, extra_info=dict(extra))
        idx = [0, b]                                       # one conditional, one unconditional sample of the batch
        ctx = torch.cat([c2[16 * i:16 * (i + 1)] for i in idx])
        ref = unet_forward(sd, spec, x_in[idx], t_in[idx].long(), ctx, dict(EXTRA_INFO))
        eps_err = [rel(eps[i], ref[k]) for k, i in enumerate(idx)]
        lat = sampler_call(*dev_in)                        # the timed call, once more
        cond = (dev_in[0][:16], ["p"], dict(EXTRA_INFO))
        uncond = (dev_in[1][:16], [""], dict(EXTRA_INFO))
        apply = lambda x, t, c: unet_forward(sd, spec, x, t, c[0], dict(c[2]))
        ref_lat, _ = ddim_sample(apply, DDIM_STEPS, [1, 4, LATENT, LATENT], cond, uncond, GUIDANCE, dev_in[2][:1])
        lat_err = rel(lat[0], ref_lat[0])
        out["parity"] = {"eps_rel_l2": {"cond_sample_0": eps_err[0], f"uncond_sample_{b}": eps_err[1]}, "eps_budget": 1e-2,
                         "final_latent_rel_l2_image0": lat_err, "latent_budget": 2e-2,
                         "ok": bool(max(eps_err) < 1e-2 and lat_err < 2e-2),
                         "against": "fp32 oracle port (oracle/unet_oracle.py, pinned to the unmodified reference by "
                                    "tests/golden) in eager torch on this GPU, TF32 off"}
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = tf32

        def time_step(autocast_dtype):
            def run():
                if autocast_dtype is None:
                    return unet_forward(sd, spec, x_in, t_in.long(), c2, dict(EXTRA_INFO))
                with torch.autocast("cuda", dtype=autocast_dtype):
                    return unet_forward(sd, spec, x_in, t_in.long(), c2, dict(EXTRA_INFO))
            run()
            torch.cuda.synchronize()
            ts = []
            for _ in range(3):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); run(); e1.record(); torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1))
            return sorted(ts)[1]

        base = {"fp32_ms": time_step(None), "bf16_autocast_ms": time_step(torch.bfloat16),
                "fp16_autocast_ms": time_step(torch.float16)}
        base.update({"unit": "ms per UNet step, batch 16, 64x64 latent", "kind": "port",
                     "what": "oracle port of the reference modules (same torch ops the reference issues: F.conv2d, "
                             "F.linear, einsum attention with the [B*8, N, N] scores materialised, F.group_norm) run "
                             "eagerly on this B200 through cuDNN / cuBLAS; fp16 autocast is the reference CLI's default "
                             "(scripts/stable_txt2img.py:179-184,614)"})
        out["gpu_eager_baseline"] = base
    del sd
    torch.cuda.empty_cache()
    return out


def train_leg(dev, unet, world, rank, steps):
    """Stage-1 distillation (BASELINE.json configs[3]) through train_cond.Stage1Trainer: per GPU 4 x 2 accumulation
    micro-batches at 64x64 latents, one NCCL all-reduce of the gradient bucket per optimizer step, clip 0.5, Prodigy."""
    import torch
    import torch.distributed as dist
    from adaprompt_b200.synthetic import stage1_batch, stage1_stack
    from adaprompt_b200.train_cond import Stage1Trainer
    step, params = stage1_stack(dev, unet=unet)
    trainer = Stage1Trainer(step, params, world_size=world, accum=2)
    g = torch.Generator().manual_seed(100 + rank)
    batches = lambda: [stage1_batch(dev, 4, LATENT, g) for _ in range(2)]
    for _ in range(2):
        trainer.optimizer_step(batches())
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        out = trainer.optimizer_step(batches())
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    trainer.optimizer_step(batches(), time_allreduce=True)
    ms_step = float(ms) / steps
    n_params = sum(p.numel() for p in params)
    info = {"metric": "stage1_distill_samples_per_sec", "value": world * 8 / (ms_step / 1e3), "unit": "samples/s",
            "ms_per_optimizer_step": ms_step, "optimizer_steps": steps, "allreduce_ms": trainer.allreduce_ms,
            "allreduce_bytes_per_step": 4 * trainer.bucket.flat.numel() if world > 1 else 0,
            "collective": "one NCCL all-reduce (SUM -> mean) of the flat fp32 gradient bucket per optimizer step" if world > 1 else None,
            "trainable_params": n_params, "loss": float(out["loss"]), "grad_norm": float(out["grad_norm"]),
            "config": {"workload": "stage1_distill_bs4x2accum_64x64", "micro_batch": 4, "grad_accum": 2,
                       "optimizer": "Prodigy", "clip_grad_norm": 0.5, "cuda_graph": "one graph per optimizer step",
                       "execution": "the 2 x 4 samples of the accumulation loop run through the conditioning and the frozen UNet as one "
                                    "batch of 8 (same gradient of sum_k MSE_k / 2; tests/test_train_gpu.py compares with the loop)",
                       "teacher_eps": "fixed random tensor (SURVEY.md 8(d) config 4)"}}
    del trainer, step, params
    torch.cuda.empty_cache()
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-vae", action="store_true", help="skip the sampling + first-stage-decoder leg (vae_decode key)")
    ap.add_argument("--breakdown", action="store_true", help="print the per-kernel-class table to stderr")
    ap.add_argument("--no-train", action="store_true", help="skip the Stage-1 training leg (train_step key)")
    ap.add_argument("--no-parity", action="store_true", help="skip the parity gate / GPU eager baseline legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of each leg returned (rank 0) as DIR/<name>.npy: the sampler's "
                         "samples and intermediates, the decoded images, the training step's loss and gradient norm")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    # stdout carries exactly ONE line (the JSON record): anything a library prints there (NCCL's version banner on the
    # first communicator, ...) is sent to stderr for the duration of the run
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(line: dict):
        os.write(json_fd, (json.dumps(line) + "\n").encode())

    if args.impl == "reference":
        return run_reference(args, emit)

    import torch
    import torch.distributed as dist
    from adaprompt_b200 import _lib
    from adaprompt_b200.ddim import DDIMSampler
    from adaprompt_b200.ldm_lite import SD15_UNET_CONFIG, LatentDiffusionLite
    from adaprompt_b200.unet import UNetModel
    from adaprompt_b200.weights import spec_of, synth_state_dict

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the B200 path has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep stdout to the ONE JSON line
        dist.init_process_group("nccl", device_id=dev)

    # ---- model: random-init SD-1.5 architecture, same recipe as the parity tests ---------------------
    with torch.device("meta"):
        unet = UNetModel(**SD15_UNET_CONFIG)
    unet = unet.to_empty(device=dev)
    unet.load_state_dict(synth_state_dict(spec_of(unet), 1234))
    unet.eval().prepare()
    model = LatentDiffusionLite(unet).to(dev)
    sampler = DDIMSampler(model, use_cuda_graph=not args.no_graph)

    b = IMAGES_PER_GPU
    g = torch.Generator().manual_seed(42 + rank)
    host = {  # pinned host copies of one step's inputs (e2e leg)
        "c": torch.randn(16 * b, 77, 768, generator=g).pin_memory(),
        "uc": torch.randn(16 * b, 77, 768, generator=g).pin_memory(),
        "x_T": torch.randn(b, 4, LATENT, LATENT, generator=g).pin_memory(),
    }
    out_host = torch.empty(b, 4, LATENT, LATENT).pin_memory()
    prompts = ["a photo of a z, , , , , , , , , , , , , , , "] * b
    extra = {"use_layerwise_context": True, "use_conv_attn_kernel_size": -1, "placeholder2indices": None,
             "is_training": False}

    def sample(c, uc, x_T):
        """-> (samples, intermediates), what DDIMSampler.sample returns to its caller."""
        cond = (c, prompts, dict(extra))
        uncond = (uc, [""] * b, dict(extra))
        return sampler.sample(DDIM_STEPS, b, [4, LATENT, LATENT], conditioning=cond,
                              unconditional_conditioning=uncond, guidance_scale=GUIDANCE, eta=0.0, x_T=x_T,
                              verbose=False)

    def one_call(c, uc, x_T):
        return sample(c, uc, x_T)[0]

    def fresh_device_inputs():
        return host["c"].to(dev), host["uc"].to(dev), host["x_T"].to(dev)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, n):
        """n calls bracketed by barrier + synchronize; CUDA events on the current stream; max over ranks."""
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        sync_all()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # ---- value: inputs resident in HBM -------------------------------------------------------------------
    resident = {}          # the result of the latest call (--dump-outputs writes the last timed one)

    def step_resident():
        # new context tensors per call => the per-prompt K/V projection cache is rebuilt inside the timed
        # region (SURVEY.md section 8(d): "KV cache warm-up included"); clones are device-to-device.
        resident["out"] = sample(dev_in[0].clone(), dev_in[1].clone(), dev_in[2])

    dev_in = fresh_device_inputs()
    for _ in range(max(3, args.warmup)):
        step_resident()
    launches0 = _lib.TRACE.count + sampler.graph_kernel_launches
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    ms_total = timed(step_resident, args.steps)
    launches = _lib.TRACE.count + sampler.graph_kernel_launches - launches0
    clock_info = clocks.stop() if rank == 0 else None
    ms_per_step = ms_total / args.steps
    value = world * b * args.steps / (ms_total / 1e3)
    dumps = {}
    if args.dump_outputs:
        samples, inter = resident.pop("out")
        dumps["samples"] = samples
        for key in ("x_inter", "pred_x0"):
            dumps.update({f"{key}_{i}": t for i, t in enumerate(inter[key])})
    resident.clear()

    # ---- e2e: host buffers in, host latents out, through the same public API ---------------------------------
    def step_e2e():
        c = host["c"].to(dev, non_blocking=True)
        uc = host["uc"].to(dev, non_blocking=True)
        x_T = host["x_T"].to(dev, non_blocking=True)
        out_host.copy_(one_call(c, uc, x_T), non_blocking=True)

    step_e2e()
    ms_e2e = timed(step_e2e, args.steps)
    e2e_value = world * b * args.steps / (ms_e2e / 1e3)
    h2d = sum(t.numel() * t.element_size() for t in host.values())
    d2h = out_host.numel() * out_host.element_size()

    # ---- row N1 (SURVEY.md 8(f)): the same call followed by the first-stage decoder (latents -> 512x512 RGB) -----
    vae_info = None
    if not args.no_vae:
        from adaprompt_b200.vae import AutoencoderKL
        with torch.device("meta"):
            vae = AutoencoderKL()
        vae = vae.to_empty(device=dev)
        vae.load_state_dict(synth_state_dict(spec_of(vae), 4321))
        vae.eval()
        model.first_stage_model = vae
        rgb_host = torch.empty(b, 3, 8 * LATENT, 8 * LATENT).pin_memory()
        lat = one_call(*dev_in)
        for _ in range(2):
            model.decode_first_stage(lat)
        ms_dec = timed(lambda: model.decode_first_stage(lat), args.steps) / args.steps

        def step_e2e_rgb():
            c = host["c"].to(dev, non_blocking=True)
            uc = host["uc"].to(dev, non_blocking=True)
            x_T = host["x_T"].to(dev, non_blocking=True)
            rgb_host.copy_(model.decode_first_stage(one_call(c, uc, x_T)), non_blocking=True)

        step_e2e_rgb()
        ms_rgb = timed(step_e2e_rgb, args.steps) / args.steps
        if args.dump_outputs:
            dumps["images"] = rgb_host.clone()
        vae_info = {"decode_ms_per_8_images": ms_dec, "decode_tflops": b * VAE_GFLOP_PER_IMAGE / 1e3 / (ms_dec / 1e3),
                    "e2e_rgb_images_per_sec": world * b / (ms_rgb / 1e3), "d2h_bytes_per_step": rgb_host.numel() * 4,
                    "note": "sampling + decode_first_stage, host prompts/noise in, host 512x512 RGB out"}
        del vae, lat
        model.first_stage_model = None
        torch.cuda.empty_cache()

    # ---- roofline of the dominant kernel: per-launch CUDA events over one eager UNet step --------------------
    peaks = measured_peaks()
    roofline, breakdown = None, None
    if rank == 0:
        x_in = torch.cat([dev_in[2]] * 2)
        t_in = torch.full((2 * b,), 501.0, device=dev)
        c2 = torch.cat([dev_in[0], dev_in[1]])
        with torch.no_grad():
            for _ in range(2):
                unet(x_in, t_in, context=c2, extra_info=dict(extra))
            with _lib.profile() as prof:
                unet(x_in, t_in, context=c2, extra_info=dict(extra))
            breakdown = prof.summary()
        step_ms = sum(v["ms"] for v in breakdown.values())
        tensor_names = ("af_conv3x3_bf16", "af_gemm_bf16", "af_attention_bf16")
        dom = max(tensor_names, key=lambda n: breakdown.get(n, {"ms": 0})["ms"])
        d = breakdown[dom]
        achieved = d["flops"] / (d["ms"] * 1e-3) / 1e12
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "r02_unet_step_traffic.json")   # one ncu pass of the same UNet step
        if not os.path.exists(tpath):
            tpath = os.path.join(ROOT, "profiles", "r01_unet_step_traffic.json")
        if os.path.exists(tpath):
            tj = json.load(open(tpath)).get(dom)
            if tj and tj["launches"]:
                traffic = tj["dram_bytes"] / tj["launches"]
                traffic_src = (f"dram__bytes_read.sum + dram__bytes_write.sum per launch, ncu pass of scripts/unet_step.py "
                               f"({os.path.relpath(tpath, ROOT)}; algorithmic {tj['algorithmic_bytes'] / tj['launches']:.3e} B)")
        roofline = {"kernel": dom, "bound": "tensor", "achieved": achieved, "peak": peaks["tflops_sustained"],
                    "unit": "TFLOP/s", "frac": achieved / peaks["tflops_sustained"], "traffic": traffic,
                    "traffic_source": traffic_src,
                    "peak_source": f"{peaks['source']} bf16 sustained (kernel timed inside a long step)",
                    "launches": d["launches"], "avg_launch_ms": d["ms"] / d["launches"],
                    "share_of_unet_step": d["ms"] / step_ms,
                    "how": "CUDA events around every launch of one eager UNet step (batch 16, t=501)"}
        gn_parts = [breakdown[n] for n in ("af_groupnorm_silu", "af_groupnorm_apply", "af_groupnorm_finalize",
                                           "af_groupnorm_stats") if n in breakdown]
        if gn_parts:
            # the whole GroupNorm class: apply + finalize + stats launches; bytes = 6 per element (fp32 in, bf16 out),
            # charged once (to the apply pass); also reported against the 4 B/element of a bf16-in / bf16-out norm
            gn_ms = sum(v["ms"] for v in gn_parts)
            gn_bytes = sum(v["bytes"] for v in gn_parts)
            gbs = gn_bytes / (gn_ms * 1e-3) / 1e9
            ap_ = breakdown.get("af_groupnorm_apply") or breakdown.get("af_groupnorm_silu")
            big = prof.by_shape.get(f"groupnorm_apply B{2 * b} HW{LATENT * LATENT} C320")
            roofline["groupnorm_silu"] = {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                          "frac": gbs / peaks["hbm_gbs"], "share_of_unet_step": gn_ms / step_ms,
                                          "launches": sum(v["launches"] for v in gn_parts), "ms": gn_ms,
                                          "bytes_per_element": 6,
                                          "frac_at_4_bytes_per_element": gbs * 4 / 6 / peaks["hbm_gbs"],
                                          "apply_pass_only_gbs": ap_["bytes"] / (ap_["ms"] * 1e-3) / 1e9 if ap_ else None,
                                          "apply_64x64_c320_gbs": big["bytes"] / (big["ms"] * 1e-3) / 1e9 if big else None}
        at = breakdown.get("af_attention_bf16")
        if at:
            tf = at["flops"] / (at["ms"] * 1e-3) / 1e12
            roofline["attention"] = {"bound": "tensor", "achieved": tf, "peak": peaks["tflops_sustained"],
                                     "unit": "TFLOP/s", "frac": tf / peaks["tflops_sustained"],
                                     "share_of_unet_step": at["ms"] / step_ms}
            hot = prof.by_shape.get(f"attention_bf16 B{2 * b} Nq{LATENT * LATENT} Nk{LATENT * LATENT} d40")
            if hot and hot["ms"] > 0:      # the long-sequence self-attention launches alone (3/4 of the class's time)
                htf = hot["flops"] / (hot["ms"] * 1e-3) / 1e12
                roofline["attention"]["self_attention_64x64_d40"] = {
                    "launches": hot["launches"], "ms_each": hot["ms"] / hot["launches"], "achieved": htf,
                    "frac": htf / peaks["tflops_sustained"]}
        for cls, key in (("af_conv3x3_bf16", "conv3x3"), ("af_gemm_bf16", "gemm")):
            v = breakdown.get(cls)
            if v and v["ms"] > 0:          # both tensor-core classes, whichever of them is the dominant kernel above
                ctf = v["flops"] / (v["ms"] * 1e-3) / 1e12
                roofline[key] = {"bound": "tensor", "achieved": ctf, "peak": peaks["tflops_sustained"], "unit": "TFLOP/s",
                                 "frac": ctf / peaks["tflops_sustained"], "launches": v["launches"],
                                 "share_of_unet_step": v["ms"] / step_ms}
        roofline["unet_step_ms_eager_sum"] = step_ms
        if args.breakdown:
            for n, v in sorted(breakdown.items(), key=lambda kv: -kv[1]["ms"]):
                tf = v["flops"] / (v["ms"] * 1e-3) / 1e12 if v["ms"] > 0 else 0
                gb = v["bytes"] / (v["ms"] * 1e-3) / 1e9 if v["ms"] > 0 else 0
                print(f"{n:24s} launches {v['launches']:4d}  {v['ms']:8.3f} ms  {tf:8.1f} TFLOP/s  {gb:8.1f} GB/s",
                      file=sys.stderr)
            for n, v in sorted(prof.by_shape.items(), key=lambda kv: -kv[1]["ms"])[:60]:
                tf = v["flops"] / (v["ms"] * 1e-3) / 1e12 if v["ms"] > 0 else 0
                gb = v["bytes"] / (v["ms"] * 1e-3) / 1e9 if v["ms"] > 0 else 0
                print(f"  {n:52s} x{v['launches']:3d} {v['ms']:8.3f} ms  {tf:7.1f} TF/s {gb:7.1f} GB/s", file=sys.stderr)

    # ---- parity gate + practical GPU baseline (rank 0) -------------------------------------------------------
    oracle_legs = {}
    if rank == 0 and not args.no_parity:
        oracle_legs = gpu_oracle_legs(dev, unet, one_call, dev_in, extra, b)

    # ---- Stage-1 training leg (all ranks: its gradient all-reduce is the one data-path collective) ------------
    train_info = None
    if not args.no_train:
        sampler.__dict__.pop("_step_graphs", None)
        sampler._graphs = {}
        torch.cuda.empty_cache()
        train_info = train_leg(dev, unet, world, rank, args.steps)
        if args.dump_outputs:
            dumps.update({f"train_{k}": torch.tensor(train_info[k], dtype=torch.float64) for k in ("loss", "grad_norm")})

    # ---- CPU baseline (rank 0, N = 1 only): the oracle port on the host cores, bounded sample ---------------
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        med, times, cores = cpu_oracle_pair_seconds(6, 1)
        cpu_baseline = {"value": 1.0 / (DDIM_STEPS * med), "unit": "images/s", "cores": cores, "kind": "port",
                        "sample": f"{len(times)} x one CFG-pair UNet forward (batch 2, 64x64 latent, fp32 oracle), "
                                  f"median {med:.2f} s; one image = 50 such steps"}

    if rank == 0:
        unet_tflops = (2 * b * UNET_GFLOP_PER_SAMPLE * DDIM_STEPS / 1e3) / (ms_per_step / 1e3)
        line = {
            "metric": "ddim50_cfg_512x512_images_per_sec", "value": value, "unit": "images/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": workload_config(world, graph=not args.no_graph),
            "unet_step_ms": ms_per_step / DDIM_STEPS,
            "unet_tflops_algorithmic": unet_tflops,
            "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches,
            "vae_decode": vae_info,
            "clocks": clock_info,
            "roofline": roofline,
            "cpu_baseline": cpu_baseline,
            "parity": oracle_legs.get("parity"),
            "gpu_eager_baseline": oracle_legs.get("gpu_eager_baseline"),
            "train_step": train_info,
        }
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, dumps)
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
