"""Time the CLIP ResNet fine-tuning step (CLIPResNetTrainPlan): the CLIP RN50 image encoder at 224^2, batch 64 per GPU, bf16, a cosine
distillation loss to fixed unit targets on the embedding; forward and backward + optimizer captured as two CUDA graphs around the
loss (one rank; several ranks run eagerly with the bucketed NCCL all-reduce).  Prints one JSON line shaped like bench.py's
`train_step` record, with the GPU name and power limit read in the same run.

  python scripts/time_train_clip.py [--steps 20 --warmup 3]
  python scripts/time_train_clip.py --profile OUT.json    # separate run: torch.profiler kernel-time shares of eager steps
"""
import argparse
import json
import os
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bcos_b200  # noqa: E402,F401
from bcos_b200.engine import CLIPResNetTrainPlan  # noqa: E402
from bcos_b200.models import clip_rn_state_shapes  # noqa: E402
from bcos_b200.utils import dist as D  # noqa: E402
from bcos_b200.utils import synth  # noqa: E402
from time_train_densenet import gpu_info  # noqa: E402

# kernels of the attention-pool head (csrc/bcosk_head.cu), and the fused pool backward of the trunk (csrc/bcosk_train.cu)
HEAD_KERNELS = ("sgemm_batched_kernel", "head_tokens_kernel", "row_softmax_kernel", "softmax_bwd_kernel", "seed_from_tokens_kernel")
POOL_KERNELS = ("pool_bwd_norm_kernel",)


def profile(plan: CLIPResNetTrainPlan, loss_fn, steps: int, path: str) -> dict:
    from torch.profiler import ProfilerActivity, profile as tprof
    for _ in range(2):
        plan.train_step(None, loss_fn)
    torch.cuda.synchronize()
    with tprof(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            plan.train_step(None, loss_fn)
        torch.cuda.synchronize()
    per = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0:
            per[e.key] = per.get(e.key, 0.0) + t / steps / 1e3       # ms per step
    total = sum(per.values())
    head = {k: v for k, v in per.items() if any(n in k for n in HEAD_KERNELS)}
    pool = {k: v for k, v in per.items() if any(n in k for n in POOL_KERNELS)}
    top = sorted(per.items(), key=lambda kv: -kv[1])[:15]
    out = {"kernel_ms_per_step": total, "head_ms_per_step": sum(head.values()), "head_share": sum(head.values()) / total,
           "pool_bwd_ms_per_step": sum(pool.values()), "head_kernels": dict(sorted(head.items(), key=lambda kv: -kv[1])),
           "top_kernels_ms": dict(top)}
    with open(path, "w") as fh:
        json.dump(out, fh, indent=1)
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--size", type=int, default=224)
    ap.add_argument("--dtype", default="bf16", choices=("bf16", "fp16"))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--profile", default=None, help="write torch.profiler kernel shares of eager steps to this file instead of timing")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_train_clip.py measures on a CUDA device (B200); there is nothing to time without one")
    rank, local, world = D.env_rank()
    torch.cuda.set_device(local)
    D.init("nccl")
    dev = f"cuda:{local}"
    sd = synth.synthetic_checkpoint("clip_rn50", clip_rn_state_shapes())
    plan = CLIPResNetTrainPlan(sd, a.batch, dtype=a.dtype, device=dev, image_size=a.size, world_size=world,
                               loss_scale=1024.0 if a.dtype == "fp16" else 1.0)
    targets = F.normalize(torch.randn(a.batch, plan.emb.shape[1], generator=torch.Generator().manual_seed(7 + rank)), dim=1).to(dev)

    def loss_fn(emb):
        return (1 - F.cosine_similarity(emb, targets, dim=1)).mean()

    plan.x_in.copy_(torch.from_numpy(synth.synth_images_u8(a.batch, a.size, 3000 + rank)).to(dev))
    if a.profile:
        out = profile(plan, loss_fn, max(a.steps, 1), a.profile)
        if rank == 0:
            print(json.dumps({**gpu_info(local), "arch": "clip_rn50", "batch_per_gpu": a.batch, **{k: v for k, v in out.items() if k != "top_kernels_ms"}}))
        D.barrier()
        return
    captured = plan.capture()
    losses = [float(plan.train_step(None, loss_fn)) for _ in range(max(a.warmup, 1))]
    D.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.steps):
        plan.train_step(None, loss_fn)
    e1.record()
    D.barrier()
    ms = D.max_over_ranks(e0.elapsed_time(e1)) / a.steps
    losses.append(float(plan.last_loss))
    rec = {"workload": f"B-cosification fine-tuning step of the CLIP RN50 image encoder at {a.size}^2 (cosine distillation loss on the "
                       "embedding), batch-sharded backward, NCCL gradient all-reduce",
           **gpu_info(local), "batch_per_gpu": a.batch, "n_gpus": world, "steps": a.steps, "ms_per_step": ms,
           "value": world * a.batch / (ms * 1e-3), "unit": "img/s", "dtype": f"{a.dtype} operands, fp32 head / accumulate / master weights / optimizer state",
           "tflops_per_gpu": plan.train_flops() / (ms * 1e-3) / 1e12, "launches_per_step": plan.num_train_launches(),
           "cuda_graph": "forward + backward/optimizer (two graphs around the torch loss)" if captured else False,
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
