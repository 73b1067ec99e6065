"""Host logic of the CLIP ResNet fine-tuning plan on CPU: the stem's operand index map, gradient slots, buckets, the gloo all-reduce
(world size 2)."""
import os
import subprocess
import sys

import pytest
import torch

import bcos_oracle as OR
from bcos_b200.engine import CLIPResNetTrainPlan
from bcos_b200.engine import pack as P
from bcos_b200.utils import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEAD = ["model.attnpool.c_proj.linear.weight", "model.attnpool.v_proj.weight", "model.attnpool.k_proj.weight", "model.attnpool.q_proj.weight"]


@pytest.fixture(scope="module")
def rn50():
    sd = synth.synth_state_dict(OR.clip_rn_state_shapes(), 0)
    return sd, CLIPResNetTrainPlan(sd, 2, device="cpu", image_size=64)


def _gathered(plan, lay):
    _, idx = plan._fwd_pack_of(lay)
    return torch.where(idx >= 0, plan.w_flat[idx.clamp(min=0).long()], torch.zeros(()))


def test_operand_index_maps_reproduce_the_packing(rn50):
    """the 3x3/2 stem conv's 2x2/1 space-to-depth operand gathered from w_flat is the packing of stem_s2d_weight of the 3x3 master
    weight; the other stem convs and a pooled block's convs map back to theirs"""
    sd, plan = rn50
    want, _ = P.pack_b(P.fwd_weight_taps(P.stem_s2d_weight(sd["model.conv1.linear.weight"], 32)), 1, 32, torch.float32)
    assert torch.equal(_gathered(plan, plan.stem), want)
    s2, s3 = plan.stem_convs[1:]
    for lay, key in ((s2, "model.conv2"), (s3, "model.conv3")):
        wt, _ = plan._even_taps(P.fwd_weight_taps(sd[key + ".linear.weight"]), P.conv_taps(3, 3), 32)   # 9 taps -> whole K stages
        w, _ = P.pack_b(wt, 1, 32, torch.float32)
        assert torch.equal(_gathered(plan, lay), w), key
    blk = plan.blocks[3]                                          # layer2.0: anti-aliasing pool and pooled downsample
    assert blk.name == "model.layer2.0" and blk.stride == 2 and blk.t2p is not None and blk.xp is not None
    for lay in blk.convs + [blk.ds]:
        key = lay.name + (".linear.weight" if lay is not blk.ds else ".1.linear.weight")
        w, _ = P.pack_b(P.fwd_weight_taps(sd[key]), 1, 64, torch.float32)
        assert torch.equal(_gathered(plan, lay), w), lay.name


def test_gradient_slots_are_a_bijection_over_the_trainable_keys(rn50):
    sd, plan = rn50
    gi = plan.gidx.long()
    assert gi.numel() == plan.w_flat.numel() and gi.unique().numel() == gi.numel() and int(gi.min()) >= 0
    assert int(gi.max()) + 1 == plan.g_flat.numel()
    shapes = OR.clip_rn_state_shapes()
    keys = {k for k in shapes if k.endswith(".weight")}             # conv / BN weights and the head's q, k, v, c_proj
    assert set(plan.gradients()) == keys and set(plan.state_dict()) == keys | {k for k in shapes if k.endswith(".running_var")}
    # the head's matrices: identity slots, one AGC unit per output row
    C = plan.trunk_out.c
    for key in HEAD:
        hw = [h for h in plan.head_w.values() if h.key == key][0]
        assert torch.equal(gi[hw.w_off:hw.w_off + hw.c], hw.gbn_off + torch.arange(hw.c))
        assert hw.cols == C and hw.rows == shapes[key][0]
    offs = plan.unit_off.cpu()
    cols = plan.unit_cols.cpu()
    n_head = sum(h.rows for h in plan.head_w.values())
    assert offs.numel() == sum(l.fwd.n + (l.bn is not None) for l in plan.layers) + n_head and bool((cols[-n_head:] == C).all())
    assert int(cols.to(torch.int64).sum()) == plan.w_flat.numel()


def test_bucket_order(rn50):
    """the buckets tile the gradient buffer in backward order: the head first (c_proj, v, k, q), the stem last"""
    _, plan = rn50
    assert plan.buckets[0][0] == 0 and plan.buckets[-1][1] == plan.g_flat.numel()
    assert all(a[1] == b[0] for a, b in zip(plan.buckets, plan.buckets[1:]))
    offs = [[h for h in plan.head_w.values() if h.key == k][0].gbn_off for k in HEAD]
    assert offs == sorted(offs) and offs[0] == 0
    last = plan.blocks[-1].convs
    assert max(offs) < last[2].g_off < last[1].g_off < last[0].g_off
    s1, s2, s3 = plan.stem_convs
    assert max(l.g_off for b in plan.blocks for l in b.convs) < s3.g_off < s2.g_off < s1.g_off
    names = [o.name for o in plan.bwd_ops]
    assert names.index("attnpool.tokens.bwd.q") < names.index("attnpool.seed") < names.index("model.layer4.2.conv3.bwd.reduce")
    assert names.index("model.layer2.0.avgpool.bwd") < names.index("model.layer2.0.conv2.bwd.reduce")
    assert names[-1].startswith("allreduce[") and "stem.conv1.dgrad" not in names


def test_only_b2_is_built():
    sd = synth.synth_state_dict(OR.clip_rn_state_shapes((1, 1, 1, 1)), 0)
    with pytest.raises(ValueError):
        CLIPResNetTrainPlan(sd, 2, layers=(1, 1, 1, 1), device="cpu", image_size=64, b=1.0)


def test_bucketed_allreduce_gloo_world2():
    code = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, %r)
sys.path.insert(0, os.path.join(%r, "oracle"))
import bcos_oracle as OR
from bcos_b200.engine import CLIPResNetTrainPlan
from bcos_b200.utils import synth
rank = int(os.environ["RANK"])
dist.init_process_group("gloo", rank=rank, world_size=2)
sd = synth.synth_state_dict(OR.clip_rn_state_shapes(), 0)
plan = CLIPResNetTrainPlan(sd, 2, device="cpu", image_size=64, world_size=2, bucket_mb=25.0)
assert len(plan.buckets) >= 3
plan.g_flat.fill_(float(rank + 1))
for a, b in plan.buckets:
    plan._allreduce(a, b)
assert bool((plan.g_flat == 3.0).all())
dist.destroy_process_group()
print("ALLREDUCE_OK", rank)
""" % (ROOT, ROOT)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29547")
    procs = [subprocess.Popen([sys.executable, "-c", code], env=dict(env, RANK=str(r)), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
             for r in range(2)]
    outs = [p.communicate(timeout=300)[0] for p in procs]
    assert all("ALLREDUCE_OK" in o for o in outs), outs
