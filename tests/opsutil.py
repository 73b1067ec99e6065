"""Helpers for the GPU parity tests: move launch records between devices and compare their outputs; the launch list of every plan
(`plan_ops`), from which the fp64 kernel tests collect their geometries."""
from __future__ import annotations

import dataclasses
import functools
from typing import Dict, Iterable

import torch
from torch import Tensor

from bcos_b200.engine import ops as O


@functools.lru_cache(maxsize=None)
def plan_ops():
    """[(tag, op)] of the forward and backward launches of the plans, built on the host at batch 1 (only shapes are read): the
    inference plans of every model family (ResNet-50 at 224 / 448 in both modes and input formats, DenseNet-121 / -169, CLIP RN50
    with both heads, ViT-Ti at 224 / 256, CLIP ViT) and the fine-tuning steps of ResNet-50 and DenseNet-121 at 224."""
    from bcos_b200.engine import CLIPViTPlan, DenseNetPlan, DenseNetTrainPlan, ResNetPlan, ResNetTrainPlan, ViTPlan
    from bcos_b200.engine.clip_rn import CLIPResNetPlan
    from bcos_b200.models import (clip_rn_state_shapes, clip_vit_state_shapes, densenet_state_shapes, resnet_state_shapes,
                                  vit_state_shapes)
    from bcos_b200.utils import synth
    out = []
    sd50 = synth.synth_state_dict(resnet_state_shapes("resnet50"), 0)
    for size in (224, 448):
        for mode in ("parity", "throughput"):
            for u8 in (False, True):
                p = ResNetPlan("resnet50", sd50, 1, mode=mode, device="cpu", image_size=size, input_u8=u8, want_rgba=True)
                out += [(f"resnet50@{size}/{mode}/{'u8' if u8 else 'f32'}", op) for op in p.fwd_ops + p.bwd_ops]
    for arch in ("densenet121", "densenet169"):
        p = DenseNetPlan(arch, synth.synth_state_dict(densenet_state_shapes(arch), 0), 1, mode="parity", device="cpu")
        out += [(f"{arch}@224", op) for op in p.fwd_ops + p.bwd_ops]
    csd = synth.synth_state_dict(clip_rn_state_shapes(), 0)
    for fused in (True, False):
        p = CLIPResNetPlan(csd, 1, mode="parity", device="cpu", fused_head=fused)
        out += [(f"clip_rn50@224/{'fused' if fused else 'module'}_head", op) for op in p.fwd_ops + p.bwd_ops]
    vsd = synth.synth_state_dict(vit_state_shapes("simple_vit_ti_patch16_224"), 0)
    for size in (224, 256):
        p = ViTPlan("simple_vit_ti_patch16_224", vsd, 1, mode="parity", device="cpu", image_size=size)
        out += [(f"vit_ti@{size}", op) for op in p.fwd_ops + p.bwd_ops]
    csd = synth.synth_state_dict(clip_vit_state_shapes(224, 32, 128, 2, 64), 0)
    p = CLIPViTPlan(csd, 1, heads=2, mode="parity", device="cpu")
    out += [("clip_vit_b32@224", op) for op in p.fwd_ops + p.bwd_ops]
    p = ResNetTrainPlan("resnet50", sd50, 1, device="cpu")
    out += [("train/resnet50@224", op) for op in p.fwd_ops + p.bwd_ops]
    p = DenseNetTrainPlan("densenet121", synth.synth_state_dict(densenet_state_shapes("densenet121"), 0), 1, device="cpu")
    out += [("train/densenet121@224", op) for op in p.fwd_ops + p.bwd_ops]
    return out


def ops_of(kind):
    """[(tag, op)] of `plan_ops()` whose launch record is a `kind`"""
    return [(tag, op) for tag, op in plan_ops() if isinstance(op, kind)]


OUTPUT_FIELDS = {
    O.IgemmOp: ["y", "gain", "maskbits", "sq_out", "out2", "amax"],
    O.InputPrepOp: ["out", "sq"],
    O.PatchNormOp: ["inv_norm"],
    O.AvgPoolFwdOp: ["y", "sq"],
    O.AvgPoolBwdMulOp: ["gx"],
    O.GapLogitsOp: ["logits", "pred"],
    O.FcSeedOp: ["out1", "out2"],
    O.ContribMapOp: ["cmap", "grad6"],
    O.ExplanationImageOp: ["out"],
    O.TrunkOutOp: ["out"],
    O.SeedFromNchwOp: ["out1", "out2"],
    O.VitPatchifyOp: ["out", "sq"],
    O.VitContribMapOp: ["cmap", "grad6"],
    O.VitLnFwdOp: ["y", "rstd", "sq"],
    O.VitLnBwdOp: ["G_out", "ghat"],
    O.VitGeluFwdOp: ["a", "sq", "gain"],
    O.VitAttentionOp: ["out"],
    O.PixelSqsumOp: ["sq"],
    O.DenseBnReluFwdOp: ["y", "sq", "maskbits"],
    O.DenseBnReluBwdOp: ["G"],
    O.DenseSliceCastOp: ["out"],
    O.CopyChannelsOp: ["dst"],
    O.StemIm2colOp: ["out", "inv_norm"],
    O.SgemmOp: ["c"],
    O.HeadTokensOp: ["tokens"],
    O.RowSoftmaxOp: ["s"],
    O.SeedFromTokensOp: ["out1", "out2"],
}


def to_device(op, device, memo: Dict[int, Tensor] | None = None):
    """Copy a launch record; tensors are cloned to `device` (aliasing preserved through `memo`)."""
    memo = {} if memo is None else memo
    changes = {}
    for f in dataclasses.fields(op):
        v = getattr(op, f.name)
        if isinstance(v, Tensor):
            if id(v) not in memo:
                base = v._base
                if base is not None:
                    # a view (interior of a zero-bordered buffer, or a reshaped alias of another operand): move the whole
                    # buffer once and keep the view, so that aliasing between launch records survives the copy
                    if id(base) not in memo:
                        memo[id(base)] = base.detach().clone().to(device)
                    memo[id(v)] = memo[id(base)].as_strided(v.shape, v.stride(), v.storage_offset())
                else:
                    memo[id(v)] = v.detach().clone().to(device)
            changes[f.name] = memo[id(v)]
    return dataclasses.replace(op, **changes)


def max_rel_err(a: Tensor, b: Tensor) -> float:
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    denom = b.abs().max().clamp_min(1e-30)
    return ((a - b).abs().max() / denom).item()


def _planes_of(op, name: str) -> int:
    if isinstance(op, O.IgemmOp):
        return {"y": 1 if op.y_f32 else op.y_planes, "out2": op.out2_planes}.get(name, 1)
    if name in ("out", "y", "gx", "out1", "out2") and hasattr(op, "planes"):
        return op.planes
    return 1


def _join(t: Tensor, planes: int) -> Tensor:
    c = t.shape[-1] // planes
    return sum(t[..., p * c:(p + 1) * c].double() for p in range(planes))


def compare(op_ref, op_dev, tol: float, fields: Iterable[str] | None = None) -> Dict[str, float]:
    errs = {}
    for name in (fields or OUTPUT_FIELDS[type(op_ref)]):
        r, d = getattr(op_ref, name), getattr(op_dev, name)
        if r is None:
            continue
        planes = _planes_of(op_ref, name)
        if planes > 1 and r.dtype not in (torch.int32, torch.int64, torch.float32):
            r, d = _join(r.cpu(), planes), _join(d.cpu(), planes)
        if r.dtype in (torch.int32, torch.int64, torch.uint8):
            mism = (r.cpu() != d.cpu()).float().mean().item()
            errs[name] = mism
            # ReLU decisions / kept MaxOut units of values that tie to the last bit may fall the other way
            assert mism <= (2e-3 if name in ("maskbits", "amax") else 0.0), (op_ref.name, name, mism)
        else:
            e = max_rel_err(d, r)
            errs[name] = e
            assert e <= tol, (op_ref.name, name, e)
    return errs


# ---------------------------------------------------------------------------------------------------------------------
# 16-bit precision planes (value = sum of the planes), for the fp64 kernel tests
# ---------------------------------------------------------------------------------------------------------------------
def store_rel(dtype: str, planes: int) -> float:
    """relative rounding of a value stored in `planes` fp16 / bf16 planes"""
    return 2.0 ** (-(11 if dtype == "fp16" else 8) * planes)


def store_floor(dtype: str, planes: int) -> float:
    """absolute floor of the same: half the fp16 subnormal spacing per plane"""
    return planes * 2.0 ** -25 if dtype == "fp16" else 0.0


def split_planes(t, planes, c):
    """[..., planes * c] 16-bit -> list of `planes` [..., c] views"""
    return [t[..., p * c:(p + 1) * c] for p in range(planes)]


def joined(t, planes, c):
    """fp64 value of [..., planes * c] 16-bit planes"""
    return sum(p.double() for p in split_planes(t, planes, c))


def check_residual_planes(t, planes, c, what):
    """every plane after the first is the round-to-nearest residual of the planes before it"""
    ps = split_planes(t, planes, c)
    for i in range(planes - 1):
        a = ps[i].abs()
        ulp = (torch.nextafter(a, torch.full_like(a, float("inf"))) - a).double()
        bad = (ps[i + 1].double().abs() > ulp / 2).sum().item()
        assert bad == 0, (what, f"plane {i + 1} is not the residual of plane {i}", bad)


def store_bound(v64, e, dtype, planes):
    """bound of a stored value whose fp32 computation is within e of v64"""
    return e + store_rel(dtype, planes) * (v64.abs() + e) + store_floor(dtype, planes)
