"""Time the DenseNet fine-tuning step (DenseNetTrainPlan): DenseNet-121 at 224^2, batch 64 per GPU, bf16, the whole step captured as
one CUDA graph (one rank; several ranks run eagerly with the bucketed NCCL all-reduce).  Prints one JSON line shaped like
bench.py's `train_step` record, with the GPU name and power limit read in the same run.

  python scripts/time_train_densenet.py [--steps 20 --warmup 3]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 scripts/time_train_densenet.py
  python scripts/time_train_densenet.py --profile OUT.json    # separate run: torch.profiler kernel-time shares of eager steps
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bcos_b200  # noqa: E402,F401
from bcos_b200.engine import DenseNetTrainPlan  # noqa: E402
from bcos_b200.models import densenet_state_shapes  # noqa: E402
from bcos_b200.utils import dist as D  # noqa: E402
from bcos_b200.utils import synth  # noqa: E402

# kernels of csrc/bcosk_dense_train.cu (the DenseNet-specific batch-statistics BN and its backward)
NEW_KERNELS = ("dense_slice_stats", "dense_consumer_finalize", "dense_consumer_bwd", "dense_slice_bwd")


def gpu_info(dev: int) -> dict:
    info = {"gpu": torch.cuda.get_device_name(dev)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info.update(power_limit_w=float(q[0]), max_sm_clock_mhz=float(q[1]))
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        info.update(power_limit_w=None, max_sm_clock_mhz=None)
    return info


def profile(plan: DenseNetTrainPlan, steps: int, path: str) -> dict:
    from torch.profiler import ProfilerActivity, profile as tprof
    for _ in range(2):
        plan.forward_backward()
        plan.optimizer_step()
    torch.cuda.synchronize()
    with tprof(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            plan.forward_backward()
            plan.optimizer_step()
        torch.cuda.synchronize()
    per = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0:
            per[e.key] = per.get(e.key, 0.0) + t / steps / 1e3       # ms per step
    total = sum(per.values())
    new = {k: v for k, v in per.items() if any(n in k for n in NEW_KERNELS)}
    top = sorted(per.items(), key=lambda kv: -kv[1])[:15]
    out = {"kernel_ms_per_step": total, "new_kernels_ms_per_step": sum(new.values()), "new_kernels_share": sum(new.values()) / total,
           "new_kernels": dict(sorted(new.items(), key=lambda kv: -kv[1])), "top_kernels_ms": dict(top)}
    with open(path, "w") as fh:
        json.dump(out, fh, indent=1)
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--arch", default="densenet121")
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--size", type=int, default=224)
    ap.add_argument("--dtype", default="bf16", choices=("bf16", "fp16"))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--profile", default=None, help="write torch.profiler kernel shares of eager steps to this file instead of timing")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_train_densenet.py measures on a CUDA device (B200); there is nothing to time without one")
    rank, local, world = D.env_rank()
    torch.cuda.set_device(local)
    D.init("nccl")
    dev = f"cuda:{local}"
    sd = synth.synthetic_checkpoint(a.arch, densenet_state_shapes(a.arch))
    plan = DenseNetTrainPlan(a.arch, sd, a.batch, dtype=a.dtype, device=dev, image_size=a.size, world_size=world,
                             loss_scale=65536.0 if a.dtype == "fp16" else 1.0)
    imgs = torch.from_numpy(synth.synth_images_u8(a.batch, a.size, 2000 + rank)).to(dev)
    labels = (torch.arange(a.batch) * 37 + rank) % 1000
    plan.load_batch(imgs, labels.to(dev))
    if a.profile:
        out = profile(plan, max(a.steps, 1), a.profile)
        if rank == 0:
            print(json.dumps({**gpu_info(local), "arch": a.arch, "batch_per_gpu": a.batch, **{k: v for k, v in out.items() if k != "top_kernels_ms"}}))
        D.barrier()
        return
    captured = plan.capture()
    losses = [float(plan.train_step()) for _ in range(max(a.warmup, 1))]
    D.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.steps):
        plan.train_step()
    e1.record()
    D.barrier()
    ms = D.max_over_ranks(e0.elapsed_time(e1)) / a.steps
    losses.append(float(plan.loss))
    rec = {"workload": f"B-cosification fine-tuning step of {a.arch} at {a.size}^2, batch-sharded backward, NCCL gradient all-reduce",
           **gpu_info(local), "batch_per_gpu": a.batch, "n_gpus": world, "steps": a.steps, "ms_per_step": ms,
           "value": world * a.batch / (ms * 1e-3), "unit": "img/s", "dtype": f"{a.dtype} operands, fp32 accumulate / master weights / optimizer state",
           "tflops_per_gpu": plan.train_flops() / (ms * 1e-3) / 1e12, "launches_per_step": plan.num_train_launches(), "cuda_graph": bool(captured),
           "collective": None if world == 1 else f"NCCL all_reduce(sum) of {len(plan.buckets)} fp32 gradient buckets on a side stream, overlapped with the backward pass",
           "allreduce_bytes_per_step": 0 if world == 1 else int(plan.g_flat.numel() * 4),
           "loss_first_steps": losses[:3], "loss_last": losses[-1], "loss_decreases_on_fixed_batch": bool(losses[-1] < losses[0])}
    if rank == 0:
        print(json.dumps(rec))
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
