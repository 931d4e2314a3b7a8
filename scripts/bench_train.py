"""Stage-1 distillation step timing (BASELINE.json configs[3]): per GPU batch 4 x 2 gradient-accumulation micro-steps,
64x64 latent, UNet forward + activation backward (one CUDA graph), SubjBasisGenerator (12-layer trainable CLIP text
model) forward / backward with weight gradients, frozen CLIP, one all-reduce of the flat gradient bucket per optimizer
step (NCCL over NVLink when launched with torchrun, N > 1), clip by norm 0.5, Prodigy.  Synthetic data, random-init
weights; the teacher's eps is a fixed random tensor (SURVEY.md section 8(d) config 4).  One JSON line on rank 0.

    python scripts/bench_train.py [--steps 3] [--warmup 2] [--bs 4] [--accum 2] [--no-graph] [--breakdown]
    python scripts/bench_train.py --masked [--steps 3] [--warmup 2]    (image-masked vs unmasked batches, see masked())
    python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 scripts/bench_train.py
"""
import argparse
import json
import os
import sys
import time

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--bs", type=int, default=4)
    ap.add_argument("--accum", type=int, default=2)
    ap.add_argument("--latent", type=int, default=64)
    ap.add_argument("--no-graph", action="store_true", help="eager autograd tape instead of the CUDA graph")
    ap.add_argument("--unet-graph", action="store_true", help="only the UNet forward + backward as a graph (round-2 first form)")
    ap.add_argument("--loop-unet", action="store_true", help="step graph with the UNet run per micro-batch instead of fused")
    ap.add_argument("--breakdown", action="store_true", help="per-entry-point CUDA-event times of one optimizer step (stderr)")
    ap.add_argument("--masked", action="store_true", help="time image-masked against unmasked optimizer steps and the "
                    "masked against the unmasked fused attention backward (one GPU)")
    args = ap.parse_args()
    if args.masked:
        return masked(args)
    import torch.distributed as dist
    from adaprompt_b200 import _lib
    from adaprompt_b200.synthetic import stage1_batch, stage1_stack
    from adaprompt_b200.train_cond import Stage1Trainer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep stdout to the ONE JSON line
        dist.init_process_group("nccl", device_id=dev)
    step, params = stage1_stack(dev)
    n_params = sum(p.numel() for p in params)
    trainer = Stage1Trainer(step, params, world_size=world, accum=args.accum, use_graph=False if args.no_graph else (True if args.unet_graph else "step"))
    if args.loop_unet and trainer._gstep is not None:
        trainer._gstep.fuse_unet = False
    g = torch.Generator().manual_seed(100 + rank)

    def optimizer_step(time_allreduce=False):
        return trainer.optimizer_step([stage1_batch(dev, args.bs, args.latent, g) for _ in range(args.accum)],
                                      time_allreduce=time_allreduce)

    for _ in range(args.warmup):
        out = optimizer_step()
    torch.cuda.synchronize()
    if args.breakdown and rank == 0:
        # the fused step = one eager pass over bs x accum samples (what the step graph holds)
        fused = not (args.no_graph or args.unet_graph or args.loop_unet)
        eager = Stage1Trainer(step, params, world_size=1, accum=1 if fused else args.accum, use_graph=False,
                              optimizer=trainer.optimizer)
        batches = ([stage1_batch(dev, args.bs * args.accum, args.latent, g)] if fused else
                   [stage1_batch(dev, args.bs, args.latent, g) for _ in range(args.accum)])
        eager.optimizer_step(batches)
        with _lib.profile() as prof:
            eager.optimizer_step(batches)
        summ = prof.summary()
        tot = sum(v["ms"] for v in summ.values())
        print(f"one EAGER optimizer step: {sum(v['launches'] for v in summ.values())} C-ABI calls, {tot:.1f} ms of kernel time", file=sys.stderr)
        for n, v in sorted(summ.items(), key=lambda kv: -kv[1]["ms"])[:24]:
            print(f"  {n:28s} x{v['launches']:5d} {v['ms']:8.2f} ms  {v['flops'] / max(v['ms'], 1e-9) / 1e9:7.1f} TFLOP/s", file=sys.stderr)
        for n, v in sorted(prof.by_shape.items(), key=lambda kv: -kv[1]["ms"])[:40]:
            print(f"    {n:60s} x{v['launches']:4d} {v['ms']:8.2f} ms", file=sys.stderr)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(args.steps):
        out = optimizer_step()
    e1.record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_step = float(ms) / args.steps
    optimizer_step(time_allreduce=True)
    peak_gb = torch.cuda.max_memory_allocated() / 2 ** 30
    if rank == 0:
        print(json.dumps({"metric": "stage1_distill_samples_per_sec", "value": world * args.bs * args.accum / (ms_step / 1e3),
                          "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                          "ms_per_optimizer_step": ms_step, "wall_ms_per_step": wall * 1e3 / args.steps,
                          "allreduce_ms": trainer.allreduce_ms,
                          "config": {"workload": "stage1_distill_bs4x2accum_64x64", "micro_batch": args.bs,
                                     "grad_accum": args.accum, "latent": [4, args.latent, args.latent],
                                     "trainable_params": n_params, "optimizer": "Prodigy", "clip_grad_norm": 0.5,
                                     "cuda_graph": "none" if args.no_graph else ("unet" if args.unet_graph else "optimizer step"),
                                     "micro_batches_fused_through_unet": not (args.no_graph or args.unet_graph or args.loop_unet),
                                     "allreduce_bytes_per_step": 4 * n_params if world > 1 else 0},
                          "loss": float(out["loss"]), "grad_norm": float(out["grad_norm"]),
                          "prodigy_d": trainer.optimizer.param_groups[0]["d"],
                          "peak_memory_gib": peak_gb, "dtype": "bf16 operands / fp32 residual stream and gradients",
                          "data": "synthetic", "scaling": "weak"}))
    if world > 1:
        dist.destroy_process_group()


def masked(args):
    """Cost of image masks: optimizer steps on batches with img_mask / fg_mask (synthetic.synthetic_masks) and without,
    alternated step by step in one process; then CUDA-event times of the fused attention backward at N = 4096, d = 40,
    B = 8, 8 heads with an all-kept and a 50 % random key mask, alternated.
    A trainer keeps one step graph, recaptured when the mask set changes, so each kind has its own trainer; both share
    one optimizer (Prodigy binds the parameters into its own buffer at its first step).  That first step moves the
    parameter storage, which is part of the capture key, so each trainer captures twice: in warm-up steps 1 and 2."""
    if args.warmup < 2:
        raise SystemExit("--masked needs --warmup >= 2: each trainer captures its step graph in warm-up steps 1 and 2")
    from adaprompt_b200 import ops
    from adaprompt_b200.packing import head_pad
    from adaprompt_b200.synthetic import stage1_batch, stage1_stack
    from adaprompt_b200.train_cond import Stage1Trainer
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    step, params = stage1_stack(dev)
    plain = Stage1Trainer(step, params, accum=args.accum, use_graph="step")
    trainers = {"plain": plain,
                "masked": Stage1Trainer(step, params, accum=args.accum, use_graph="step", optimizer=plain.optimizer)}
    g = torch.Generator().manual_seed(100)
    ms = {"plain": [], "masked": []}
    for it in range(args.warmup + args.steps):
        for kind, tr in trainers.items():
            batches = [stage1_batch(dev, args.bs, args.latent, g, masks=kind == "masked") for _ in range(args.accum)]
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            tr.optimizer_step(batches)
            e1.record()
            e1.synchronize()
            if it >= args.warmup:
                ms[kind].append(e0.elapsed_time(e1))
    # the fused backward kernels alone
    B, N, h, d = 8, 4096, 8, 40
    dp = head_pad(d)
    gk = torch.Generator(device="cpu").manual_seed(1)

    def rnd(*shape, scale=1.0):
        return (torch.randn(*shape, generator=gk) * scale).to(torch.bfloat16).to(dev)

    q, k, vp, dop = rnd(B * N, h * dp, scale=0.2), rnd(B * N, h * dp), rnd(B * N, h * dp), rnd(B * N, h * dp)
    qT, kT, dOT = (t.t().contiguous() for t in (q, k, dop))
    lse = torch.full((B, h, N), 14.0, device=dev)
    delta = torch.zeros(B, h, N, device=dev)
    kms = {"plain": None, "masked": (torch.rand(B, N, generator=gk) < 0.5).to(torch.uint8).to(dev)}
    kern = {"plain": [], "masked": []}
    reps = 20
    for it in range(6):
        for kind, km in kms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                ops.attention_bwd(q, k, vp, dop, qT, kT, dOT, lse, delta, B=B, heads=h, N=N, d=d, key_mask=km)
            e1.record()
            e1.synchronize()
            if it >= 1:
                kern[kind].append(e0.elapsed_time(e1) / reps)
    name = torch.cuda.get_device_name(dev)
    try:
        import subprocess
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:  # noqa: BLE001
        power = "unknown"
    med = lambda v: sorted(v)[len(v) // 2]
    print(json.dumps({"metric": "stage1_masked_vs_unmasked", "device": name, "power_limit": power,
                      "config": {"micro_batch": args.bs, "grad_accum": args.accum, "latent": args.latent,
                                 "cuda_graph": "optimizer step"},
                      "ms_per_optimizer_step": {k: med(v) for k, v in ms.items()},
                      "ms_per_optimizer_step_all": ms,
                      "fused_attention_bwd_ms": {k: med(v) for k, v in kern.items()},
                      "fused_attention_bwd_shape": {"B": B, "N": N, "heads": h, "d": d, "kept_keys": "all / 50 % random"},
                      "fused_attention_bwd_ms_all": kern}))


if __name__ == "__main__":
    main()
