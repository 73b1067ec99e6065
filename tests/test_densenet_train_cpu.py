"""Host logic of the DenseNet fine-tuning plan on CPU: operand index maps, gradient slots, buckets, the gloo all-reduce (world size 2)."""
import os
import subprocess
import sys

import torch

import bcos_oracle as OR
from bcos_b200.engine import DenseNetTrainPlan
from bcos_b200.engine import pack as P
from bcos_b200.engine.densenet import dn_names
from bcos_b200.models import densenet_state_shapes
from bcos_b200.utils import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARCH = "densenet121"


def _plan(**kw):
    sd = synth.synth_state_dict(densenet_state_shapes(ARCH), 0)
    return sd, DenseNetTrainPlan(ARCH, sd, 2, device="cpu", image_size=64, **kw)


def _gathered(plan, lay):
    _, idx = plan._fwd_pack_of(lay)
    return torch.where(idx >= 0, plan.w_flat[idx.clamp(min=0).long()], torch.zeros(()))


def test_operand_index_maps_reproduce_the_packing():
    """every packed forward operand (stem, conv1, conv2, transition, classifier) gathered from w_flat is the ordinary packing of the
    state-dict weight"""
    sd, plan = _plan()
    nm = dn_names(4)
    want0, _ = P.pack_b(P.fwd_weight_taps(P.stem_s2d_weight(sd[nm["conv0"] + ".linear.weight"], 32)), 1, 32, torch.float32)
    assert torch.equal(_gathered(plan, plan.stem), want0)
    blk = plan.blocks[1]
    n1, c1, c2 = blk.layers[2]                        # C_l = 128 + 2 * 32 = 192: a prefix that is not a multiple of 128
    assert n1.c == 192
    convs = [c1, c2, plan.blocks[0].t_conv, plan.blocks[2].t_conv, plan.fc]
    for lay in convs:
        key = (lay.name if lay is not plan.fc else "model.classifier") + ".linear.weight"
        want, _ = P.pack_b(P.fwd_weight_taps(sd[key]), 1, 64, torch.float32)
        assert torch.equal(_gathered(plan, lay), want), lay.name


def test_gradient_slots_and_buckets():
    sd, plan = _plan()
    gi = plan.gidx.long()
    assert gi.numel() == plan.w_flat.numel() and gi.unique().numel() == gi.numel() and int(gi.min()) >= 0
    assert int(gi.max()) < plan.g_flat.numel()
    # the buckets tile the gradient buffer in backward order: classifier first, norm5 next, the stem last
    assert plan.buckets[0][0] == 0 and plan.buckets[-1][1] == plan.g_flat.numel()
    assert all(a[1] == b[0] for a, b in zip(plan.buckets, plan.buckets[1:]))
    assert plan.fc.g_off == 0 and plan.norm5.gbn_off == plan.fc.fwd.n * plan.fc.fwd.ktot
    last = plan.blocks[-1].layers[-1]
    assert last[1].g_off < last[0].gbn_off < plan.blocks[-1].layers[-2][2].g_off
    assert plan.stem.g_off > max(n.gbn_off for n in plan.norms)
    # a BN weight gradient slot per consumer norm, and the gradient keys are the reference's trainable parameters
    assert len(plan.norms) == sum(plan.block_cfg) + len(plan.block_cfg)
    keys = {k for k, v in OR.densenet_state_shapes(ARCH).items() if k.endswith(".linear.weight") or (k.endswith(".weight") and len(v) == 1)}
    assert set(plan.gradients()) == keys
    # every consumer owns its running variance
    assert all(n.name in plan.running_var for n in plan.norms)


def test_bucketed_allreduce_gloo_world2():
    code = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, %r)
from bcos_b200.engine import DenseNetTrainPlan
from bcos_b200.models import densenet_state_shapes
from bcos_b200.utils import synth
rank = int(os.environ["RANK"])
dist.init_process_group("gloo", rank=rank, world_size=2)
sd = synth.synth_state_dict(densenet_state_shapes("densenet121"), 0)
plan = DenseNetTrainPlan("densenet121", sd, 2, device="cpu", image_size=64, world_size=2, bucket_mb=8.0)
assert len(plan.buckets) >= 3
plan.g_flat.fill_(float(rank + 1))
for a, b in plan.buckets:
    plan._allreduce(a, b)
assert bool((plan.g_flat == 3.0).all())
dist.destroy_process_group()
print("ALLREDUCE_OK", rank)
""" % ROOT
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29541")
    procs = [subprocess.Popen([sys.executable, "-c", code], env=dict(env, RANK=str(r)), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
             for r in range(2)]
    outs = [p.communicate(timeout=300)[0] for p in procs]
    assert all("ALLREDUCE_OK" in o for o in outs), outs
