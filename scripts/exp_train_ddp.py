"""2+ ranks (torchrun): the bucketed NCCL all-reduce inside ResNetTrainPlan (DenseNetTrainPlan with --arch densenet121,
CLIPResNetTrainPlan with --arch clip_rn50 and a cosine loss on the embedding) gives the
SUM of the ranks' local gradients, the ranks end a step with identical weights, and the timing of a step with / without the collective.
  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29517 scripts/exp_train_ddp.py [--arch A]"""
import argparse, os, sys, json
import torch, torch.distributed as dist
import torch.nn.functional as F
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bcos_b200  # noqa
from bcos_b200.engine import CLIPResNetTrainPlan, DenseNetTrainPlan, ResNetTrainPlan
from bcos_b200.models import clip_rn_state_shapes, densenet_state_shapes, resnet_state_shapes
from bcos_b200.utils import synth, dist as D

ap = argparse.ArgumentParser()
ap.add_argument("--arch", default="resnet50", help="resnet18/34/50, densenet121/169/201 or clip_rn50")
arch = ap.parse_args().arch
clip = arch == "clip_rn50"
if clip:
    Plan, shapes = (lambda a, sd, B, **kw: CLIPResNetTrainPlan(sd, B, **kw)), (lambda a: clip_rn_state_shapes())
else:
    Plan, shapes = (DenseNetTrainPlan, densenet_state_shapes) if arch.startswith("densenet") else (ResNetTrainPlan, resnet_state_shapes)

rank, local, world = D.env_rank()
torch.cuda.set_device(local)
D.init("nccl")
dev = f"cuda:{local}"
B = 32
sd = synth.synthetic_checkpoint(arch, shapes(arch))
imgs = torch.from_numpy(synth.synth_images_u8(B, 224, 500 + rank)).to(dev)
labels = ((torch.arange(B) * 13 + rank * 7) % 1000).to(dev)
targets = F.normalize(torch.randn(B, 1024, generator=torch.Generator().manual_seed(13 + rank)), dim=1).to(dev)


def loss_fn(emb):
    return (1 - F.cosine_similarity(emb, targets, dim=1)).mean()


def load(p):
    if clip:
        p.x_in.copy_(imgs)
    else:
        p.load_batch(imgs, labels)


def fwd_bwd(p):
    if clip:
        p.forward_backward(loss_fn)
    else:
        p.forward_backward()


def step(p):
    if clip:
        p.train_step(None, loss_fn)
    else:
        p.train_step()


local_plan = Plan(arch, sd, B, device=dev, world_size=1)
load(local_plan)
fwd_bwd(local_plan)
g_own = local_plan.g_flat.clone()
g_local = g_own.clone()
dist.all_reduce(g_local)
plan = Plan(arch, sd, B, device=dev, world_size=world, bucket_mb=25.0)
load(plan)
fwd_bwd(plan)
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
        step(p)
    D.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        step(p)
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
