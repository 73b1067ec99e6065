"""2+ ranks (torchrun): the bucketed NCCL all-reduce inside ResNetTrainPlan (DenseNetTrainPlan with --arch densenet121) gives the
SUM of the ranks' local gradients, the ranks end a step with identical weights, and the timing of a step with / without the collective.
  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29517 scripts/exp_train_ddp.py [--arch A]"""
import argparse, os, sys, json
import torch, torch.distributed as dist
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bcos_b200  # noqa
from bcos_b200.engine import DenseNetTrainPlan, ResNetTrainPlan
from bcos_b200.models import densenet_state_shapes, resnet_state_shapes
from bcos_b200.utils import synth, dist as D

ap = argparse.ArgumentParser()
ap.add_argument("--arch", default="resnet50", help="resnet18/34/50 or densenet121/169/201")
arch = ap.parse_args().arch
Plan, shapes = (DenseNetTrainPlan, densenet_state_shapes) if arch.startswith("densenet") else (ResNetTrainPlan, resnet_state_shapes)

rank, local, world = D.env_rank()
torch.cuda.set_device(local)
D.init("nccl")
dev = f"cuda:{local}"
B = 32
sd = synth.synthetic_checkpoint(arch, shapes(arch))
imgs = torch.from_numpy(synth.synth_images_u8(B, 224, 500 + rank)).to(dev)
labels = ((torch.arange(B) * 13 + rank * 7) % 1000).to(dev)
local_plan = Plan(arch, sd, B, device=dev, world_size=1)
local_plan.load_batch(imgs, labels)
local_plan.forward_backward()
g_own = local_plan.g_flat.clone()
g_local = g_own.clone()
dist.all_reduce(g_local)
plan = Plan(arch, sd, B, device=dev, world_size=world, bucket_mb=25.0)
plan.load_batch(imgs, labels)
plan.forward_backward()
torch.cuda.synchronize()
rel = float((plan.g_flat - g_local).norm() / g_local.norm())
per_bucket = [(float((plan.g_flat[a:b] - g_local[a:b]).norm() / g_local[a:b].norm()), float((plan.g_flat[a:b] - g_own[a:b]).norm() / g_own[a:b].norm()))
              for a, b in plan.buckets]
print("rank", rank, "per bucket (vs sum, vs own):", per_bucket, flush=True)
plan.optimizer_step()
w = plan.w_flat.clone()
w0 = w.clone()
dist.broadcast(w0, 0)
same_t = torch.tensor([1.0 if torch.equal(w, w0) else 0.0], device=dev)
dist.all_reduce(same_t, op=dist.ReduceOp.MIN)
same = bool(same_t.item() == 1.0)
def timed(p, n=6):
    for _ in range(2):
        p.train_step()
    D.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        p.train_step()
    e1.record()
    D.barrier()
    return D.max_over_ranks(e0.elapsed_time(e1)) / n
t_ddp = timed(plan)
t_local = timed(local_plan)
if rank == 0:
    print(json.dumps({"world": world, "arch": arch, "batch_per_gpu": B, "buckets": len(plan.buckets), "allreduce_MB": plan.g_flat.numel() * 4 / 1e6,
                      "grad_sum_rel_err_vs_manual_allreduce": rel, "weights_identical_across_ranks": same,
                      "ms_per_step_with_allreduce": t_ddp, "ms_per_step_local_only": t_local}))
D.shutdown()
