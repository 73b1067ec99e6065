"""Fused execution plan for B-cosified ResNets: forward + dynamic-linear explanation.

Network (reference): `BcosifyNetwork(ResNetBcos(...))` bcosify.py:22-53 on the torchvision skeleton with
FC-before-GAP (bcos/models/standard_models.py:36-54), maxpool -> AvgPool2d(3,2,1) and all biases removed
(bcos/experiments/ImageNet/bcosification/model.py:47-55).  Explanation: `BcosUtilMixin.explain`
bcos/common.py:92-188 evaluated for the whole batch at once (images are independent in eval mode).

Every conv+BN(+residual)+ReLU group is ONE `bcosk_igemm` launch (tcgen05 implicit GEMM, fused epilogue);
the explanation pass is the chain of explain-dgrad launches whose epilogues multiply by the producer
layer's saved gain, so no stand-alone element-wise pass touches an activation-sized tensor except the two
poolings.  Data layout in HBM: NHWC, 16-bit, optional precision planes (see engine/pack.py).
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Tuple

import torch
from torch import Tensor

from .. import _lib as L
from . import ops as O
from . import pack as P
from .base import Act, BlockRec, ConvRec, PlanBase

IMAGENET_MEAN_ADDINVERSE = (0.485, 0.456, 0.406, 0.515, 0.544, 0.594)  # reference bcosify.py:14
IMAGENET_STD_ADDINVERSE = (0.229, 0.224, 0.225, 0.229, 0.224, 0.225)   # reference bcosify.py:15

RESNET_ARCH = {
    "resnet18": ("basic", [2, 2, 2, 2]),
    "resnet34": ("basic", [3, 4, 6, 3]),
    "resnet50": ("bottleneck", [3, 4, 6, 3]),
    "resnet101": ("bottleneck", [3, 4, 23, 3]),
}


# Operand formats of a plan (DESIGN.md section 4 holds the measured accuracy / cost of each against the reference):
#   parity          two fp16 planes + fp32-faithful accumulation in the forward pass, one fp16 plane in the (linear)
#                   explanation pass, seed gradient scaled by 4096: meets the whole parity contract (argmax, logits 2e-3,
#                   map cosine 0.999, max-abs 1e-3 of the map range).  THE DEFAULT.
#   parity_full     two fp16 planes everywhere (the explanation pass too)
#   throughput      one bf16 plane (the format BASELINE.json names): fastest, does NOT meet the map tolerances on random-init
#                   deep nets (argmax may flip where two logits are closer than the rounding noise) - opt-in
#   throughput_fp16 one fp16 plane: same speed, keeps argmax / logits / cosine >= 0.998
PRECISION_MODES = {
    "parity": dict(planes=2, dtype="fp16", explain_planes=1, seed_scale=4096.0),
    "parity_full": dict(planes=2, dtype="fp16", explain_planes=2, seed_scale=4096.0),
    "throughput": dict(planes=1, dtype="bf16", explain_planes=1, seed_scale=1.0),
    "throughput_fp16": dict(planes=1, dtype="fp16", explain_planes=1, seed_scale=4096.0),
}


def resolve_precision(mode: Optional[str], planes: Optional[int], dtype: Optional[str], explain_planes: Optional[int],
                      seed_scale: Optional[float]) -> Dict[str, object]:
    """Named mode -> (planes, dtype, explain_planes, seed_scale).  Explicit planes / dtype arguments select a format by
    hand (then unspecified fields take the historical defaults: one bf16 plane, unscaled seed)."""
    if planes is None and dtype is None:
        cfg = dict(PRECISION_MODES[mode or "parity"])
    else:
        if mode is not None:
            raise ValueError("pass either `mode` or explicit planes / dtype, not both")
        cfg = dict(planes=1 if planes is None else int(planes), dtype=dtype or "bf16", explain_planes=None, seed_scale=1.0)
    if explain_planes is not None:
        cfg["explain_planes"] = int(explain_planes)
    if seed_scale is not None:
        cfg["seed_scale"] = float(seed_scale)
    return cfg


class ResNetPlan(PlanBase):
    def __init__(self, arch: str, state_dict: Dict[str, Tensor], batch: int, *, mode: Optional[str] = None,
                 planes: Optional[int] = None, dtype: Optional[str] = None,
                 device="cuda", image_size: int = 224, explain: bool = True, want_grad6: bool = False, b: float = 2.0,
                 bn_eps: float = 1e-5, mean=IMAGENET_MEAN_ADDINVERSE, std=IMAGENET_STD_ADDINVERSE,
                 logit_bias: Optional[float] = -math.log(1000 - 1), logit_temperature: Optional[float] = None,
                 seed_scale: Optional[float] = None, stem_kch: int = 32, input_u8: bool = False, want_rgba: bool = False,
                 rgba_smooth: int = 15, rgba_percentile: float = 99.5, explain_planes: Optional[int] = None):
        cfg = resolve_precision(mode, planes, dtype, explain_planes, seed_scale)
        planes, dtype, explain_planes, seed_scale = cfg["planes"], cfg["dtype"], cfg["explain_planes"], cfg["seed_scale"]
        self.precision = cfg
        super().__init__(batch, planes=planes, dtype=dtype, device=device, explain=explain, b=b, bn_eps=bn_eps,
                         state_dict=state_dict, explain_planes=explain_planes)
        self.arch = arch
        self.kind, self.layers = RESNET_ARCH[arch]
        self.mean, self.std = tuple(mean), tuple(std)
        self.inv_std = tuple(1.0 / s for s in std)
        self.logit_bias = 0.0 if logit_bias is None else float(logit_bias)
        self.inv_temp = 1.0 if logit_temperature is None else 1.0 / float(logit_temperature)
        self.seed_scale = float(seed_scale)
        self.stem_kch = stem_kch
        self.stem_cp = 32 if stem_kch == 32 else 64
        self.size = image_size
        self.input_u8 = input_u8
        self.want_rgba, self.rgba_smooth, self.rgba_percentile = want_rgba, rgba_smooth, rgba_percentile
        self.blocks: List[BlockRec] = []
        self._build_forward()
        if explain:
            self._build_explain(want_grad6 or want_rgba)

    def _build_forward(self) -> None:
        nb, S, pl = self.nb, self.size, self.planes
        sd = self.sd
        # network input: fp32 [nb,6,S,S] = [x, 1-x], or uint8 RGB [nb,3,S,S] (inverse channels formed on the fly)
        self.x_in = self._empty(nb, 3, S, S, dtype=torch.uint8) if self.input_u8 else self._empty(nb, 6, S, S, dtype=torch.float32)
        # ---- stem: normalise + space-to-depth, 7x7/2 conv as a 4x4/1 conv, BN, ReLU
        h2 = S // 2
        # throughput mode: the stem reads a zero-bordered buffer (pad 2 before / 1 after) through one window per tile
        # (the flat window of the 4x4 space-to-depth stem spans 3 padded rows + 128 pixels: it fits two TMA boxes up to ~256^2 inputs)
        self.stem_flat = self.flat_stem and pl == 1 and not self.hp_accum and self._flat_fits(h2 + 3, 4, 16, 64, False, self.stem_kch)
        w4 = P.stem_s2d_weight(sd["model.conv1.linear.weight"], self.stem_cp)
        if self.hp_accum and self.input_u8 and self.stem_im2col:
            # contract modes with uint8 input: GEMM over the exact byte patch matrix (base.py _stem_fwd_im2col)
            y1, self.stem = self._stem_fwd_im2col("stem", self.x_in, sd["model.conv1.linear.weight"], w4, 7, 2, 3, bn="model.bn1",
                                                  mean6=self.mean, inv_std6=self.inv_std, s2d_pad=(2, 1), stem_cp=self.stem_cp)
        else:
            a0 = self._padded(nb, h2, h2, self.stem_cp, 2, 1) if self.stem_flat else self._empty(nb, h2, h2, pl * self.stem_cp)
            sq0 = self._empty(1, nb * S * S, dtype=torch.float32)
            self.fwd_ops.append(O.InputPrepOp("input_prep", self.x_in, self.mean, self.inv_std, a0, self.stem_cp, pl,
                                              self.dt_code, sq0))
            # the patch norm is the ORIGINAL 7x7/2 pad-3 window over the full-resolution sums of squares
            y1, self.stem = self._conv_fwd("stem", Act(a0, self.stem_cp, sq0, 1), w4, 1, 2, 1, bn="model.bn1", relu=True,
                                           kch=self.stem_kch, want_sq=False, sq_geom=(S, S, 7, 2, 3), flat=self.stem_flat)
        # ---- AvgPool2d(3, 2, 1) (replaces maxpool)
        hp = (h2 + 2 - 3) // 2 + 1
        p1 = self._empty(nb, hp, hp, pl * 64)
        sqp = self._empty(1, nb * hp * hp, dtype=torch.float32)
        self.fwd_ops.append(O.AvgPoolFwdOp("pool", y1.t, 64, pl, 3, 2, 1, p1, self.dt_code, sqp))
        self.stem_out, self.pool_out = y1, Act(p1, 64, sqp, 1)
        x = self.pool_out
        # ---- residual stages
        exp = 1 if self.kind == "basic" else 4
        inplanes = 64
        for li, (planes_, nblocks) in enumerate(zip([64, 128, 256, 512], self.layers), start=1):
            for bi in range(nblocks):
                stride = 2 if (li > 1 and bi == 0) else 1
                pfx = f"model.layer{li}.{bi}"
                has_ds = (pfx + ".downsample.0.linear.weight") in sd
                idn, ds_rec = x, None
                if has_ds:
                    idn, ds_rec = self._conv_fwd(pfx + ".downsample", x, sd[pfx + ".downsample.0.linear.weight"], stride,
                                                 0, 0, bn=pfx + ".downsample.1", relu=False, want_sq=False)
                if self.kind == "basic":
                    t1, r1 = self._conv_fwd(pfx + ".conv1", x, sd[pfx + ".conv1.linear.weight"], stride, 1, 1,
                                            bn=pfx + ".bn1", relu=True)
                    y, r2 = self._conv_fwd(pfx + ".conv2", t1, sd[pfx + ".conv2.linear.weight"], 1, 1, 1,
                                           bn=pfx + ".bn2", relu=True, res=idn, want_mask=True)
                    recs = [r1, r2]
                else:
                    t1, r1 = self._conv_fwd(pfx + ".conv1", x, sd[pfx + ".conv1.linear.weight"], 1, 0, 0,
                                            bn=pfx + ".bn1", relu=True)
                    t2, r2 = self._conv_fwd(pfx + ".conv2", t1, sd[pfx + ".conv2.linear.weight"], stride, 1, 1,
                                            bn=pfx + ".bn2", relu=True)
                    y, r3 = self._conv_fwd(pfx + ".conv3", t2, sd[pfx + ".conv3.linear.weight"], 1, 0, 0,
                                           bn=pfx + ".bn3", relu=True, res=idn, want_mask=True)
                    recs = [r1, r2, r3]
                self.blocks.append(BlockRec(pfx, recs, ds_rec, x, y, recs[-1].mask))
                x = y
                inplanes = planes_ * exp
        # ---- classifier (1x1 B-cos conv per position) -> GAP -> LogitLayer
        wfc = sd["model.fc.linear.weight"]
        self.ncls = wfc.shape[0]
        fc, self.fc = self._conv_fwd("fc", x, wfc, 1, 0, 0, bn=None, relu=False, y_f32=True, want_sq=False)
        self.npix = x.hw[0] * x.hw[1]
        self.fc_out = fc.t.view(nb * self.npix, self.ncls)
        self.logits = self._empty(nb, self.ncls, dtype=torch.float32)
        self.pred = self._zeros(nb, dtype=torch.int32)
        self.fwd_ops.append(O.GapLogitsOp("gap_logits", self.fc_out, nb, self.npix, self.ncls, self.inv_temp,
                                          self.logit_bias, self.logits, self.pred))

    def _build_explain(self, want_grad6: bool) -> None:
        nb, pl = self.nb, self.bplanes
        for blk in self.blocks:
            for j, r in enumerate(blk.convs):
                # convs after the first get their gradient from a plain data-gradient epilogue (no shortcut terms):
                # their own strided data gradient can run as parity classes over the dense tensor
                self._alloc_ghat(r, classes=j > 0)
            if blk.ds is not None:
                self._alloc_ghat(blk.ds)
                blk.side = blk.ds.ghat
            else:
                blk.side = self._zeros(nb, blk.y.hw[0], blk.y.hw[1], pl * blk.y.c)
        self._alloc_ghat(self.stem)
        self.stem_flat_bwd = (self.flat_stem and pl == 1 and not self.bwd_hp
                              and self._flat_fits(self.stem.out_hw[1] + 3, 4, 16, 32, False))
        if self.stem_flat_bwd:     # the transposed 4x4 gather pads 1 before / 2 after
            self.stem.ghat = self._padded(nb, self.stem.out_hw[0], self.stem.out_hw[1], self.stem.cout, 1, 2)
        last = self.blocks[-1]
        assert last.ds is None, "classifier seed kernel expects an identity shortcut in the last block"
        # ---- seed: d logit[target] / d fc-input, straight through GAP and the classifier's detached scale
        c_last = last.y.c
        self.w_fc32 = self._dev(self.sd["model.fc.linear.weight"].reshape(self.ncls, c_last))
        self.bwd_ops.append(O.FcSeedOp("fc.seed", self.pred, self.fc.gain, self.w_fc32, nb, self.npix, self.ncls, c_last,
                                       self.inv_temp, self.seed_scale, last.convs[-1].gain,
                                       last.convs[-1].ghat.view(nb * self.npix, pl * c_last), last.mask,
                                       last.side.view(nb * self.npix, pl * c_last), pl, self.dt_code))
        # ---- blocks in reverse
        self.g_pool = self._zeros(nb, self.pool_out.hw[0], self.pool_out.hw[1], pl * self.pool_out.c)
        for bi in range(len(self.blocks) - 1, -1, -1):
            blk = self.blocks[bi]
            convs = blk.convs
            for j in range(len(convs) - 1, 0, -1):       # conv_j's data gradient feeds conv_{j-1}'s ghat
                m1, m1s = self._gain_of(convs[j - 1])
                self._dgrad(convs[j], y=convs[j - 1].ghat, y_map=convs[j - 1].ghat_map, mul1=m1, mul1_sqrt_scale=m1s)
            add, add_stride = blk.side, 1
            if blk.ds is not None:
                dds = self._zeros(nb, blk.ds.out_hw[0], blk.ds.out_hw[1], pl * blk.ds.cin_phys) if blk.ds.stride > 1 \
                    else self._zeros(nb, blk.x.hw[0], blk.x.hw[1], pl * blk.x.c)
                self._dgrad(blk.ds, y=dds)
                add, add_stride = dds, blk.ds.stride
            if bi > 0:
                prev = self.blocks[bi - 1]
                self._dgrad(convs[0], y=prev.convs[-1].ghat, mul1=prev.convs[-1].gain, add=add, add_stride=add_stride,
                            out2=prev.side, mul2=None if prev.ds is None else prev.ds.gain, mask2=prev.mask)
            else:
                self._dgrad(convs[0], y=self.g_pool, add=add, add_stride=add_stride)
        # ---- pool backward x stem gain, stem data gradient (space-to-depth), contribution map
        m1, m1s = self._gain_of(self.stem)
        self.bwd_ops.append(O.AvgPoolBwdMulOp("pool.bwd", self.g_pool, 64, pl, 3, 2, 1, m1, self.stem.ghat, self.dt_code, m1s))
        h2 = self.size // 2
        self.g0 = self._zeros(nb, h2, h2, self.stem_cp, dtype=torch.float32)
        self._dgrad(self.stem, y=self.g0, y_f32=True, kch=64, flat=self.stem_flat_bwd)
        self.cmap = self._zeros(nb, self.size, self.size, dtype=torch.float32)
        self.grad6 = self._zeros(nb, 6, self.size, self.size, dtype=torch.float32) if want_grad6 else None
        self.bwd_ops.append(O.ContribMapOp("contrib_map", self.g0, self.x_in, self.stem_cp, self.inv_std,
                                           1.0 / self.seed_scale, self.cmap, self.grad6))
        self.rgba = None
        if self.want_rgba:
            # the reference's published artefact: RGBA explanation images (gradient_to_image) for the whole batch
            self.rgba = self._zeros(nb, self.size, self.size, 4, dtype=torch.float32)
            tmp = self._zeros(2 * nb * self.size * self.size + nb, dtype=torch.float32)
            self.bwd_ops.append(O.ExplanationImageOp("explanation_rgba", self.grad6, self.x_in, self.rgba_smooth,
                                                     self.rgba_percentile, tmp, self.rgba))

    def load_input(self, x6: Tensor) -> None:
        """x6: [nb, 6, H, W] float32 `[x, 1-x]`, or uint8 RGB [nb, 3, H, W] for an `input_u8` plan (host or device)."""
        assert tuple(x6.shape) == tuple(self.x_in.shape), (x6.shape, self.x_in.shape)
        self.x_in.copy_(x6, non_blocking=True)

    def forward(self, x6: Optional[Tensor] = None) -> Tensor:
        if x6 is not None:
            self.load_input(x6)
        self.replay_forward()
        return self.logits

    def explain(self, x6: Optional[Tensor] = None) -> Dict[str, Tensor]:
        """Forward + explanation of each image's predicted class (argmax logit)."""
        if not self.with_explain:
            raise RuntimeError("plan was built with explain=False")
        if x6 is not None:
            self.load_input(x6)
        self.replay_all()
        out = {"logits": self.logits, "prediction": self.pred, "contribution_map": self.cmap}
        if self.grad6 is not None:
            out["dynamic_linear_weights"] = self.grad6
        if self.rgba is not None:
            out["explanation"] = self.rgba
        return out


    def explain_targets(self, x6: Optional[Tensor], targets: Tensor) -> Dict[str, Tensor]:
        """Explanations of several logits per image from ONE forward pass.

        targets: int tensor [T, nb] (class index to explain, per target set and image).  The reference recomputes the forward
        for every target (Captum InputXGradient, bcos/common.py:280-344; localisation runs 4-9 targets per grid image);
        here the forward state (gains, masks) is kept and only the explanation pass is replayed per target set.
        Returns stacked tensors: contribution_map [T, nb, H, W] (+ dynamic_linear_weights / explanation when enabled)."""
        if not self.with_explain:
            raise RuntimeError("plan was built with explain=False")
        targets = torch.as_tensor(targets)
        if targets.ndim == 1:
            targets = targets[None]
        assert targets.shape[1] == self.nb, (targets.shape, self.nb)
        # the seed kernel indexes the classifier's weights with these: reject a bad class before anything is launched
        if targets.numel() and (int(targets.min()) < 0 or int(targets.max()) >= self.ncls):
            raise ValueError(f"targets must lie in [0, {self.ncls}), got [{int(targets.min())}, {int(targets.max())}]")
        if x6 is not None:
            self.load_input(x6)
        self.replay_forward()
        pred = self.pred.clone()
        tg = targets.to(device=self.pred.device, dtype=torch.int32)
        out = {"logits": self.logits.clone(), "prediction": pred, "contribution_map": []}
        if self.grad6 is not None:
            out["dynamic_linear_weights"] = []
        if self.rgba is not None:
            out["explanation"] = []
        for t in range(tg.shape[0]):
            self.pred.copy_(tg[t])                # the seed kernel reads the class to explain from here
            self.replay_explain()
            out["contribution_map"].append(self.cmap.clone())
            if self.grad6 is not None:
                out["dynamic_linear_weights"].append(self.grad6.clone())
            if self.rgba is not None:
                out["explanation"].append(self.rgba.clone())
        self.pred.copy_(pred)
        for k in ("contribution_map", "dynamic_linear_weights", "explanation"):
            if k in out:
                out[k] = torch.stack(out[k])
        return out


class PipelinedExplainer:
    """Public end-to-end API for streams of host batches: `submit(images)` returns a ticket, `result(ticket)` the pinned
    host tensors.  Host->device copies, the CUDA-graph replay and device->host copies of consecutive batches overlap on
    three streams (copy-in, compute, copy-out) with double-buffered staging, so the steady-state cost per batch is
    max(compute, PCIe) instead of their sum.  Every batch still pays its own H2D and D2H inside the pipeline."""

    def __init__(self, plan: ResNetPlan, depth: int = 2):
        assert plan.with_explain
        if plan._graph_all is None:
            plan.capture()
        self.plan, self.depth = plan, depth
        dev = plan.device
        self.s_in, self.s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        self.s_compute = torch.cuda.current_stream(dev)
        self.d_in = [torch.empty_like(plan.x_in) for _ in range(depth)]
        self.d_logits = [torch.empty_like(plan.logits) for _ in range(depth)]
        self.d_cmap = [torch.empty_like(plan.cmap) for _ in range(depth)]
        self.h_logits = [torch.empty(plan.logits.shape, dtype=torch.float32).pin_memory() for _ in range(depth)]
        self.h_cmap = [torch.empty(plan.cmap.shape, dtype=torch.float32).pin_memory() for _ in range(depth)]
        self.ev_in = [torch.cuda.Event() for _ in range(depth)]
        self.ev_done = [torch.cuda.Event() for _ in range(depth)]
        self.ev_out = [torch.cuda.Event() for _ in range(depth)]
        self.ev_free = [torch.cuda.Event() for _ in range(depth)]     # staging input slot consumed by the compute stream
        self.count = 0

    def submit(self, host_images: Tensor) -> int:
        i = self.count
        k = i % self.depth
        if i >= self.depth:
            self.ev_out[k].synchronize()          # results of ticket i-depth have left the staging slot
        with torch.cuda.stream(self.s_in):
            if i >= self.depth:
                self.s_in.wait_event(self.ev_free[k])
            self.d_in[k].copy_(host_images, non_blocking=True)
            self.ev_in[k].record(self.s_in)
        self.s_compute.wait_event(self.ev_in[k])
        self.plan.x_in.copy_(self.d_in[k], non_blocking=True)          # device-to-device, then the slot is free again
        self.ev_free[k].record(self.s_compute)
        self.plan.replay_all()
        self.d_logits[k].copy_(self.plan.logits, non_blocking=True)
        self.d_cmap[k].copy_(self.plan.cmap, non_blocking=True)
        self.ev_done[k].record(self.s_compute)
        with torch.cuda.stream(self.s_out):
            self.s_out.wait_event(self.ev_done[k])
            self.h_logits[k].copy_(self.d_logits[k], non_blocking=True)
            self.h_cmap[k].copy_(self.d_cmap[k], non_blocking=True)
            self.ev_out[k].record(self.s_out)
        self.count += 1
        return i

    def result(self, ticket: int) -> Dict[str, Tensor]:
        k = ticket % self.depth
        assert self.count - ticket <= self.depth, "result already overwritten by a later submit"
        self.ev_out[k].synchronize()
        return {"logits": self.h_logits[k], "contribution_map": self.h_cmap[k]}

    def drain(self) -> None:
        for e in self.ev_out[: min(self.count, self.depth)]:
            e.synchronize()
