"""Fine-tuning step of a B-cosified ResNet or DenseNet (SURVEY 8f row 2, BASELINE config 5): forward in train mode, loss, full
backward, gradient all-reduce, adaptive gradient clipping + AdamW - one process per GPU, batch sharded, NCCL for the gradients.
`ResNetTrainPlan`, `DenseNetTrainPlan` and `CLIPResNetTrainPlan` (engine/clip_train.py) share `TrainPlanBase`; the DenseNet's own
kernels are described at its class.

Reference: `training_step` bcos/training/trainer.py:666-784 (outputs = model(images); loss = criterion(outputs, labels)),
autograd backward through `BcosifyConv2d.forward_impl` (bcosifyconv2d.py:50-102, scale NOT detached) and
`batch_norm_uncentered_2d` with batch statistics (batchnorm_uncentered.py:36-43), DDP gradient averaging (trainer.py:918),
`adaptive_clip_grad_` (bcos/training/agc.py:28-42), `UniformOffLabelsBCEWithLogitsLoss` (bcos/modules/losses.py:99-139).

Layout and launches.  Activations and gradients are NHWC 16-bit (bf16 by default: fp32 range, so no loss scaling); weights,
optimizer state and every per-channel / per-pixel vector are fp32.  Per conv layer
  forward   bcosk_igemm (B-cos epilogue: out = lin |lin| / n, saves the scale s and 1/n)  ->  bnu_stats / finalize / apply
  backward  train_bwd_reduce / bnu_bwd_finalize / train_bwd_apply (batch-norm + ReLU + B-cos backward in two passes)
            -> bcosk_wgrad (tcgen05, MN-major operands, split-K)  -> bcosk_igemm explain-mode data gradient (plain dgrad)
            -> sumpool_transpose (the patch-norm path, applied by the consumer of the data gradient as x * T)
The packed 16-bit operands of every launch are refreshed from the fp32 master weights with one gather launch each
(`_pack_b` records, for every operand element, the master element it comes from).  Weight gradients live in ONE flat fp32
buffer in backward order; it is all-reduced in buckets on a side stream while the backward pass continues.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Callable, Dict, List, Optional, Tuple

import torch
from torch import Tensor

from .. import _lib as L
from . import ops as O
from . import pack as P
from .base import Act, ConvRec, PlanBase
from .resnet import IMAGENET_MEAN_ADDINVERSE, IMAGENET_STD_ADDINVERSE, RESNET_ARCH


@dataclass
class FnOp:
    """A launch record that is just a bound call (everything in it goes through the C ABI or is a memset)."""
    name: str
    fn: Callable[[], None]

    def run(self) -> None:
        self.fn()


@dataclass
class WgradOp:
    """One `bcosk_wgrad` launch: dw[o, (tap, c)] += sum_m g[m, o] * x_patch[m, (tap, c)] (include/bcosk.h)."""
    name: str
    fwd: O.IgemmOp           # geometry of the forward launch
    g: Tensor                # [M, n] 16-bit
    dw: Tensor               # [n * ktot] fp32 view into the flat gradient buffer

    def params(self) -> L.WgradParams:
        f = self.fwd
        p = L.WgradParams()
        nb, h, w, ac = f.a.shape
        p.x = f.a.data_ptr()
        p.a_nb, p.a_h, p.a_w, p.a_c = nb, h, w, ac
        p.lo_w, p.lo_h = f.lo
        p.up_w, p.up_h = f.up
        p.stride_w, p.stride_h = f.stride
        p.op, p.oq = f.op, f.oq
        p.kch, p.chunks_per_tap, p.num_taps = f.kch, f.chunks_per_tap, len(f.taps)
        for i, (ow, oh) in enumerate(f.taps):
            p.tap_off_w[i], p.tap_off_h[i] = ow, oh
        p.g = self.g.data_ptr()
        p.n, p.g_ld = f.n, self.g.shape[-1]
        p.dw = self.dw.data_ptr()
        p.dtype = f.dtype
        p.split_k = 0
        return p

    def flops(self) -> float:
        return self.fwd.flops()

    def run(self) -> None:
        L.wgrad(self.params())


@dataclass
class TrainLayer:
    name: str
    rec: ConvRec
    fwd: O.IgemmOp
    x: Act                                   # input activation (a norm layer's output, the pooled stem, or the s2d image)
    out: Tensor                              # [M, o] conv output (16-bit, fp32 for the classifier)
    bn: Optional[str]                        # state-dict prefix of the norm layer that follows, None = classifier
    relu: bool
    z: Optional[Act] = None                  # norm (+ residual, ReLU) output
    res: Optional[Tensor] = None
    w_off: int = 0                           # offsets into the flat master / gradient buffers
    w_numel: int = 0
    g_off: int = 0
    bnw_off: int = -1
    gbn_off: int = -1
    alpha: Optional[Tensor] = None
    mean: Optional[Tensor] = None
    rstd: Optional[Tensor] = None
    sums: Optional[Tensor] = None
    kcoef: Optional[Tensor] = None
    s_red: Optional[Tensor] = None
    gnT: Optional[Tensor] = None
    gx: Optional[Tensor] = None              # data gradient wrt the input (16-bit, input resolution)
    need_dgrad: bool = True


class TrainPlanBase(PlanBase):
    """What the fine-tuning plans share: fp32 master weights with refreshable packed operands, the flat gradient buffer in
    backward order and its all-reduce buckets, the conv + batch-statistics BN emission and its backward, AGC + AdamW of the
    whole model, CUDA-graph capture.  Subclasses emit the network (`_build`)."""

    parity_dgrad = True          # strided 3x3 data gradients as parity classes over the dense gradient
    flat_3x3 = False             # the flat-window variants keep their weights resident: not refreshable per step here
    flat_stem = False
    fold_bn = False
    autotune_default = False

    def __init__(self, arch: str, state_dict: Dict[str, Tensor], batch: int, *, dtype: str = "bf16", device="cuda",
                 image_size: int = 224, bn_eps: float = 1e-5, bn_momentum: float = 0.1, mean=IMAGENET_MEAN_ADDINVERSE,
                 std=IMAGENET_STD_ADDINVERSE, logit_bias: Optional[float] = -math.log(1000 - 1),
                 logit_temperature: Optional[float] = None, lr: float = 1e-4, betas=(0.9, 0.999), adam_eps: float = 1e-8,
                 weight_decay: float = 0.0, agc_clip: float = 0.01, agc_eps: float = 1e-3, off_label: Optional[float] = None,
                 world_size: int = 1, bucket_mb: float = 25.0, input_u8: bool = True, loss_scale: float = 1.0):
        super().__init__(batch, planes=1, dtype=dtype, device=device, explain=True, b=2.0, bn_eps=bn_eps, state_dict=state_dict)
        self.arch = arch
        self.size, self.input_u8 = image_size, input_u8
        self.mean, self.inv_std = tuple(mean), tuple(1.0 / s for s in std)
        self.logit_bias = 0.0 if logit_bias is None else float(logit_bias)
        self.inv_temp = 1.0 if logit_temperature is None else 1.0 / float(logit_temperature)
        self.momentum = bn_momentum
        self.hyper = dict(lr=lr, beta1=betas[0], beta2=betas[1], eps=adam_eps, wd=weight_decay, clip=agc_clip, agc_eps=agc_eps)
        self.off_label = off_label
        self.world = world_size
        self.loss_scale = float(loss_scale)      # fp16 operands: gradients are carried scaled by this power of two
        self.bucket_bytes = int(bucket_mb * 1e6)
        self.step_count = 0
        self.red_blocks = 296                    # blocks (= rows of partial sums) of the per-channel reductions: two per SM
        self.layers: List[TrainLayer] = []
        self.packs: List[Tuple[Tensor, Tensor]] = []          # (packed operand, int32 source index into w_flat)
        self._cur_w_off = 0
        self._w_items: List[Tuple[str, Tensor, int]] = []     # (state-dict key, fp32 tensor, offset)
        self.norm_units: List[Tuple[int, int, int]] = []      # (master offset, gradient offset, c) of BN weights not owned by a TrainLayer
        self.row_units: List[Tuple[int, int, int, int]] = []  # (master offset, gradient offset, rows, cols) of fp32 matrices used unpacked
        self.opt_ops: List = []
        self.running_var: Dict[str, Tensor] = {}
        self.w_flat = None                    # allocated after all weights are registered (closures read self.w_flat late)
        self._build()

    # ------------------------------------------------------------------ master weights and packing
    def _register_weight(self, key: str) -> Tuple[Tensor, int]:
        """fp32 master copy of `key`; returns an INDEX-valued stand-in of the same shape (element i -> i + 1 + offset) that
        flows through the ordinary packing code, so that `_pack_b` learns where every operand element comes from."""
        w = self.sd[key]
        off = self._cur_w_off
        self._w_items.append((key, w, off))
        self._cur_w_off += w.numel()
        assert w.numel() < (1 << 24), "index stand-ins are exact in fp32 below 2^24 elements per tensor"
        return (torch.arange(w.numel(), dtype=torch.float32).view(w.shape) + 1.0), off

    def _pack_b(self, wt: Tensor, planes: int, kch: int) -> Tuple[Tensor, int]:
        idx, cpt = P.pack_b(wt, 1, kch, torch.float32)
        idx = idx.round().to(torch.int64) - 1                        # -1 = structural zero (channel / tap padding)
        idx = torch.where(idx >= 0, idx + self._pack_off, idx).to(torch.int32)   # absolute index into the flat master buffer
        buf = torch.zeros(idx.shape, dtype=self.dt, device=self.device)
        self.packs.append((buf, idx.to(self.device)))
        return buf, cpt

    # ------------------------------------------------------------------ forward
    def _conv_bn(self, name: str, x: Act, wkey: str, stride: int, pad: int, bn: Optional[str], relu: bool, res: Optional[Tensor] = None,
                 w_standin: Optional[Tensor] = None, w_off: Optional[int] = None, w_numel: Optional[int] = None,
                 pad_hi: Optional[int] = None, kch: int = 64, sq_geom=None, y_f32: bool = False, want_z_sq: bool = True,
                 y_buf: Optional[Tensor] = None, y_col: int = 0) -> TrainLayer:
        """Conv launch (+ batch-statistics BN `bn`, residual, ReLU).  `y_buf`: the conv writes columns [y_col, y_col + o) of that
        wider tensor (a DenseNet feature tensor); `out` is then a strided view."""
        if w_standin is None:
            w_standin, w_off = self._register_weight(wkey)
            w_numel = w_standin.numel()
        self._pack_off = w_off
        y, rec = self._conv_fwd(name, x, w_standin, stride, pad, pad if pad_hi is None else pad_hi, bn=None, relu=False,
                                want_sq=False, want_inv=True, kch=kch, sq_geom=sq_geom, y_f32=y_f32, y_buf=y_buf, y_col=y_col)
        fwd = self.fwd_ops[-1]
        M, o = fwd.M, fwd.n
        out = y.t.view(M, o) if y_buf is None else y_buf.view(M, -1)[:, y_col:y_col + o]
        lay = TrainLayer(name, rec, fwd, x, out, bn, relu, res=res, w_off=w_off, w_numel=w_numel)
        lay.gnT = self._empty(M, dtype=torch.float32)
        if bn is not None:
            f32 = dict(dtype=torch.float32)
            lay.alpha, lay.mean, lay.rstd = self._empty(o, **f32), self._empty(o, **f32), self._empty(o, **f32)
            # per-block partial sums (no atomics: forward statistics and the backward reduction are bit-reproducible)
            lay.sums, lay.kcoef, lay.s_red = self._empty(self.red_blocks, 2 * o, **f32), self._empty(o, **f32), self._empty(self.red_blocks, o, **f32)
            z = self._empty(*y.t.shape)
            zsq = self._empty(1, M, dtype=torch.float32) if want_z_sq else None
            lay.z = Act(z, o, zsq, 1)
            lay.bnw_off = self._cur_w_off
            self._w_items.append((bn + ".weight", self.sd[bn + ".weight"], lay.bnw_off))
            self._cur_w_off += o
            rv = self._dev(self.sd[bn + ".running_var"])
            self.running_var[bn] = rv
            dtc = self.dt_code
            self.fwd_ops.append(FnOp(name + ".bn.stats", lambda l=lay: L.bnu_stats_nhwc(l.out, l.out.shape[0], l.out.shape[1], dtc, l.sums)))
            self.fwd_ops.append(FnOp(name + ".bn.finalize", lambda l=lay, rv=rv: L.bnu_finalize(
                l.sums, l.out.shape[0], l.out.shape[1], self.w_flat[l.bnw_off:l.bnw_off + l.out.shape[1]], self.bn_eps, self.momentum, rv,
                l.alpha, l.mean, l.rstd)))
            self.fwd_ops.append(FnOp(name + ".bn.apply", lambda l=lay: L.bnu_apply_nhwc(
                l.out, l.out.shape[0], l.out.shape[1], l.alpha, l.res, l.relu, l.z.t, None if l.z.sq is None else l.z.sq, dtc)))
        self.layers.append(lay)
        return lay

    def _stem(self, conv_key: str, bn_key: str, pool_sq: bool) -> Act:
        """Input prep, the stem conv + batch-statistics BN + ReLU, the 3x3/2 average pool; returns the pooled activation."""
        nb, S = self.nb, self.size
        self.x_in = self._empty(nb, 3, S, S, dtype=torch.uint8) if self.input_u8 else self._empty(nb, 6, S, S, dtype=torch.float32)
        self.labels = self._zeros(nb, dtype=torch.int32)
        h2 = S // 2
        cp = 32
        a0 = self._empty(nb, h2, h2, cp)
        sq0 = self._empty(1, nb * S * S, dtype=torch.float32)
        self.fwd_ops.append(O.InputPrepOp("input_prep", self.x_in, self.mean, self.inv_std, a0, cp, 1, self.dt_code, sq0))
        # stem: the 7x7/2 conv as a 4x4/1 conv on the 2x2 space-to-depth input (engine/pack.py stem_s2d_weight); the stand-in goes
        # through the same linear map, so its operand elements point back at the 7x7 master weights
        w7, off7 = self._register_weight(conv_key)
        w4 = P.stem_s2d_weight(w7, cp)                                        # unmapped entries stay 0 -> index -1
        stem = self._conv_bn("stem", Act(a0, cp, sq0, 1), "", 1, 2, bn_key, True, w_standin=w4, w_off=off7, w_numel=w7.numel(),
                             pad_hi=1, kch=32, sq_geom=(S, S, 7, 2, 3), want_z_sq=False)
        stem.need_dgrad = False
        self.stem = stem
        o = stem.fwd.n
        hp = (h2 + 2 - 3) // 2 + 1
        p1 = self._empty(nb, hp, hp, o)
        sqp = self._empty(1, nb * hp * hp, dtype=torch.float32) if pool_sq else None
        self.fwd_ops.append(O.AvgPoolFwdOp("pool", stem.z.t, o, 1, 3, 2, 1, p1, self.dt_code, sqp))
        return Act(p1, o, sqp, 1)

    def _head(self, name: str, x: Act, wkey: str) -> None:
        """Classifier per position (fp32 output), global average + logit layer, UniformOffLabelsBCE and its gradient g_fc."""
        nb = self.nb
        fc = self._conv_bn(name, x, wkey, 1, 0, None, False, y_f32=True)
        self.fc = fc
        self.ncls = fc.fwd.n
        self.npix = x.hw[0] * x.hw[1]
        self.logits = self._empty(nb, self.ncls, dtype=torch.float32)
        self.pred = self._zeros(nb, dtype=torch.int32)
        self.fwd_ops.append(O.GapLogitsOp("gap_logits", fc.out, nb, self.npix, self.ncls, self.inv_temp, self.logit_bias, self.logits, self.pred))
        self.loss = self._zeros(1, dtype=torch.float32)
        self.g_fc = self._empty(nb * self.npix, self.ncls)
        off = self.off_label if self.off_label is not None else 1.0 / self.ncls
        self.fwd_ops.append(FnOp("loss.zero", self.loss.zero_))
        self.fwd_ops.append(FnOp("loss", lambda: L.bce_uniform_off(self.logits, self.labels, nb, self.ncls, off, self.inv_temp, self.npix, self.loss_scale,
                                                                  self.loss, self.g_fc, None, self.dt_code)))

    # ------------------------------------------------------------------ backward
    def _alloc_grads(self, order: List) -> None:
        """Gradient slots in backward order (`order`: TrainLayers, and norm records with `c` / `gbn_off` for BN weights that no
        TrainLayer owns), the flat gradient buffer, its zeroing launch and the bucket state."""
        g_off = 0
        for lay in order:
            if isinstance(lay, TrainLayer):
                lay.g_off = g_off
                g_off += lay.fwd.n * lay.fwd.ktot
                if lay.bn is not None:
                    lay.gbn_off = g_off
                    g_off += lay.fwd.n
            else:
                lay.gbn_off = g_off
                g_off += lay.c
        self.g_flat = self._zeros(g_off, dtype=torch.float32)
        self.buckets: List[Tuple[int, int]] = []
        self._bucket_begin = self._bucket_end = 0
        self.comm_stream = torch.cuda.Stream(self.device) if self.device.type == "cuda" else None
        self.bwd_ops.append(FnOp("grad.zero", self.g_flat.zero_))

    def _layer_bwd(self, lay: TrainLayer, ga: Tensor, gb: Optional[Tensor], tn: Optional[Tensor], ga_f32: bool = False,
                   want_gy: bool = False, gx32: Optional[Tensor] = None) -> Optional[Tensor]:
        """Emit: norm / ReLU / B-cos backward of `lay`, its weight gradient, its data gradient, its patch-norm vector.
        `gx32`: the data gradient goes to this fp32 buffer instead of a fresh 16-bit one."""
        M, o = lay.out.shape
        dtc = self.dt_code
        relu = lay.relu
        xpost = lay.z.t if (lay.z is not None and (relu or tn is not None)) else None
        out_f32 = lay.out.dtype == torch.float32
        self._alloc_ghat(lay.rec, classes=True)
        glin = lay.rec.ghat.view(M, o)
        gy = self._empty(M, o) if want_gy else None
        if lay.bn is not None:
            self.bwd_ops.append(FnOp(lay.name + ".bwd.reduce", lambda: L.train_bwd_reduce(ga, ga_f32, gb, xpost, tn, relu, lay.out, out_f32, M, o,
                                                                                         lay.s_red, dtc)))
            self.bwd_ops.append(FnOp(lay.name + ".bwd.finalize", lambda: L.bnu_bwd_finalize(
                lay.s_red, lay.rstd, self.w_flat[lay.bnw_off:lay.bnw_off + o], M, o, lay.kcoef, self.g_flat[lay.gbn_off:lay.gbn_off + o])))
        self.bwd_ops.append(FnOp(lay.name + ".bwd.apply", lambda: L.train_bwd_apply(
            ga, ga_f32, gb, xpost, tn, relu, lay.out, out_f32, lay.rec.gain, lay.alpha, lay.kcoef, lay.mean, lay.rec.inv, M, o, glin, lay.gnT,
            gy, dtc)))
        self._wgrad_dgrad(lay, glin, gx32)
        return gy

    def _wgrad_dgrad(self, lay: TrainLayer, glin: Tensor, gx32: Optional[Tensor] = None) -> None:
        """Weight gradient of `lay` from g_lin (into its slot of the flat buffer), then its data gradient."""
        o = lay.fwd.n
        self.bwd_ops.append(WgradOp(lay.name + ".wgrad", lay.fwd, glin, self.g_flat[lay.g_off:lay.g_off + o * lay.fwd.ktot]))
        self._grad_ready(lay)
        if lay.need_dgrad:
            self._pack_off = lay.w_off
            h, w = lay.rec.in_hw
            cin = lay.rec.cin_phys
            if gx32 is not None:
                assert lay.rec.stride == 1 and lay.rec.k == 1
                lay.gx = gx32
                self._dgrad(lay.rec, y=gx32, y_f32=True)
                return
            lay.gx = self._zeros(self.nb, h, w, cin)
            if lay.rec.stride > 1 and lay.rec.k == 1:
                # strided 1x1: the dense GEMM at output resolution lands on the sampled pixels of a zeroed full-resolution tensor
                s = lay.rec.stride
                self._dgrad(lay.rec, y=lay.gx, y_map=(0, h * w, s * w, s))
            else:
                self._dgrad(lay.rec, y=lay.gx)

    def _norm_path(self, lay: TrainLayer, tn: Tensor, accumulate: bool) -> None:
        """tn[input pixel] (+)= sum of lay.gnT over the windows that cover it (d ||patch|| / d x = x / ||patch||)."""
        h, w = lay.rec.in_hw
        oh, ow = lay.rec.out_hw
        k, s, pad = lay.rec.k, lay.rec.stride, lay.rec.pad_lo
        self.bwd_ops.append(FnOp(lay.name + ".normpath", lambda: L.sumpool_transpose(lay.gnT, self.nb, h, w, k, s, pad, oh, ow, accumulate, tn)))

    def _grad_ready(self, lay: TrainLayer) -> None:
        end = lay.g_off + lay.fwd.n * lay.fwd.ktot
        if lay.gbn_off >= 0:
            end = max(end, lay.gbn_off + lay.fwd.n)
        self._grad_ready_to(end)

    def _grad_ready_to(self, end: int) -> None:
        """Bucketed all-reduce: once the gradients up to `end` (backward order) fill a bucket, a side stream reduces it."""
        self._bucket_end = max(self._bucket_end, end)
        if (self._bucket_end - self._bucket_begin) * 4 >= self.bucket_bytes:
            self._close_bucket()

    def _close_bucket(self) -> None:
        a, b = self._bucket_begin, self._bucket_end
        if b > a:
            self.buckets.append((a, b))
            self.bwd_ops.append(FnOp(f"allreduce[{a}:{b}]", lambda: self._allreduce(a, b)))
            self._bucket_begin = b

    def _allreduce(self, a: int, b: int) -> None:
        """Sum g_flat[a:b] over the ranks (NCCL over NVLink on CUDA tensors; averaged later by the optimizer's 1/world).  On a
        CUDA device the collective is issued on a side stream behind an event, so the backward pass keeps running."""
        if self.world == 1:
            return
        import torch.distributed as dist
        if self.comm_stream is None:
            dist.all_reduce(self.g_flat[a:b])
            return
        ev = torch.cuda.Event()
        ev.record()
        with torch.cuda.stream(self.comm_stream):
            self.comm_stream.wait_event(ev)
            dist.all_reduce(self.g_flat[a:b])

    def _alloc_master(self) -> None:
        """flat fp32 master weights / optimizer state"""
        n_w = self._cur_w_off
        self.w_flat = self._empty(n_w, dtype=torch.float32)
        for key, w, o in self._w_items:
            self.w_flat[o:o + w.numel()].copy_(w.reshape(-1))
        self.m_flat = self._zeros(n_w, dtype=torch.float32)
        self.v_flat = self._zeros(n_w, dtype=torch.float32)

    def _build_optimizer(self) -> None:
        # ---- optimizer: gradient index of every master element (the weight-gradient kernel writes the packed layout)
        gidx = torch.full((self._cur_w_off,), -1, dtype=torch.int64)
        for lay in self.layers:
            buf, idx = self._fwd_pack_of(lay)
            idx = idx.cpu().to(torch.int64).reshape(-1)
            pos = torch.nonzero(idx >= 0).reshape(-1)
            gidx[idx[pos]] = lay.g_off + pos
            if lay.bn is not None:
                o = lay.fwd.n
                gidx[lay.bnw_off:lay.bnw_off + o] = lay.gbn_off + torch.arange(o)
        for w_off, g_off, c in self.norm_units:
            gidx[w_off:w_off + c] = g_off + torch.arange(c)
        for w_off, g_off, rows, cols in self.row_units:
            gidx[w_off:w_off + rows * cols] = g_off + torch.arange(rows * cols)
        assert int((gidx < 0).sum()) == 0, "a master weight without a gradient slot"
        self.gidx = gidx.to(torch.int32).to(self.device)
        # ---- AGC + AdamW of the WHOLE model in one launch: one unit = one output row of a conv / the whole BN weight vector
        #      (agc.py:28-42 clips unit-wise); the Adam step counter lives on the device so that the step can be a CUDA graph
        u_off, u_cols = [], []
        for lay in self.layers:
            o = lay.fwd.n
            cols = lay.w_numel // o
            u_off += [lay.w_off + i * cols for i in range(o)]
            u_cols += [cols] * o
            if lay.bn is not None:
                u_off.append(lay.bnw_off)
                u_cols.append(o)
        for w_off, _, c in self.norm_units:
            u_off.append(w_off)
            u_cols.append(c)
        for w_off, _, rows, cols in self.row_units:
            u_off += [w_off + i * cols for i in range(rows)]
            u_cols += [cols] * rows
        self.unit_off = torch.tensor(u_off, dtype=torch.int64, device=self.device)
        self.unit_cols = torch.tensor(u_cols, dtype=torch.int32, device=self.device)
        self.adam_state = self._zeros(3, dtype=torch.float32)          # {step, 1 - beta1^step, 1 - beta2^step}
        self.opt_ops.append(FnOp("adam.step", lambda: L.adam_state_step(self.adam_state, self.hyper["beta1"], self.hyper["beta2"])))
        self.opt_ops.append(FnOp("agc_adamw", self._opt_all))
        # ---- every packed 16-bit operand refreshed from the fp32 master weights in one launch
        tab = [[idx.data_ptr(), buf.data_ptr(), idx.numel()] for buf, idx in self.packs]
        self.pack_table = torch.tensor(tab, dtype=torch.int64, device=self.device)
        self.pack_max_n = max(idx.numel() for _, idx in self.packs)
        self._graph = None

    def _norm_vec(self, lay: TrainLayer) -> Tensor:
        """Patch-norm vector of `lay` at its INPUT resolution (a fresh buffer; 1x1 stride-1 layers use gnT directly)."""
        if lay.rec.k == 1 and lay.rec.stride == 1:
            return lay.gnT
        h, w = lay.rec.in_hw
        tn = self._empty(self.nb * h * w, dtype=torch.float32)
        self._norm_path(lay, tn, accumulate=False)
        return tn

    def _fwd_pack_of(self, lay: TrainLayer) -> Tuple[Tensor, Tensor]:
        for buf, idx in self.packs:
            if buf is lay.fwd.b:
                return buf, idx
        raise KeyError(lay.name)

    def _opt_all(self) -> None:
        h = self.hyper
        L.agc_adamw_multi(self.w_flat, self.g_flat, self.gidx, self.m_flat, self.v_flat, self.unit_off, self.unit_cols, self.unit_off.numel(),
                          1.0 / (self.world * self.loss_scale), h["lr"], h["beta1"], h["beta2"], h["eps"], h["wd"], h["clip"], h["agc_eps"],
                          self.adam_state)

    # ------------------------------------------------------------------ execution
    def refresh_operands(self) -> None:
        """fp32 master weights -> every packed 16-bit operand (forward, data-gradient and parity-class launches)."""
        self._require_gpu()
        L.gather_cast_multi(self.w_flat, self.pack_table, len(self.packs), self.pack_max_n, self.dt_code)

    def load_batch(self, images: Tensor, labels: Tensor) -> None:
        self.x_in.copy_(images, non_blocking=True)
        self.labels.copy_(labels.to(torch.int32), non_blocking=True)

    def forward_backward(self) -> None:
        self._require_gpu()
        O.run_ops(self.fwd_ops)
        O.run_ops(self.bwd_ops)
        if self.world > 1:
            torch.cuda.current_stream().wait_stream(self.comm_stream)

    def optimizer_step(self) -> None:
        self.step_count += 1
        O.run_ops(self.opt_ops)
        self.refresh_operands()

    def train_step(self, images: Optional[Tensor] = None, labels: Optional[Tensor] = None) -> Tensor:
        """One step: forward (train mode), loss, backward, gradient all-reduce, AGC + AdamW.  Returns the loss tensor (device)."""
        if images is not None:
            self.load_batch(images, labels)
        if self._graph is not None:
            self.step_count += 1
            self._graph.replay()
            return self.loss
        self.forward_backward()
        self.optimizer_step()
        return self.loss

    def capture(self) -> bool:
        """Capture the whole step (forward, loss, backward with the bucketed all-reduce on its side stream, AGC + AdamW, operand
        refresh: ~640 launches) as ONE CUDA graph; `train_step` replays it.  The training state (weights, moments, step counter,
        BN running variances) is saved around the warm-up steps the capture needs, so capturing does not advance training.
        Single-rank plans only: returns False (and the step stays eager) when world_size > 1."""
        self._require_gpu()
        if self.world > 1:
            # a captured graph with the NCCL all-reduce on its side stream hung on this stack (torch 2.11, NCCL 2.28.9, two B200s):
            # multi-rank steps stay eager (the whole-model optimizer / refresh launches still apply)
            return False
        state = [self.w_flat, self.m_flat, self.v_flat, self.adam_state] + list(self.running_var.values())
        keep = [t.clone() for t in state]
        steps = self.step_count

        def restore():
            for dst, src in zip(state, keep):
                dst.copy_(src)
            self.step_count = steps
            self.refresh_operands()

        side = torch.cuda.Stream(self.device)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                self.forward_backward()
                self.optimizer_step()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        restore()
        g = torch.cuda.CUDAGraph()
        try:
            with torch.cuda.graph(g):
                self.forward_backward()
                O.run_ops(self.opt_ops)
                self.refresh_operands()
        except Exception as e:  # noqa: BLE001
            import warnings
            warnings.warn(f"bcos_b200: training step not captured ({type(e).__name__}: {e}); running eagerly")
            torch.cuda.synchronize()
            restore()
            return False
        torch.cuda.synchronize()
        restore()
        self._graph = g
        return True

    # ------------------------------------------------------------------ inspection (tests, checkpoints)
    def gradients(self) -> Dict[str, Tensor]:
        """Gradients in the reference's state-dict layout (fp32), summed over ranks when world > 1."""
        out = {}
        g = self.g_flat
        for key, w, off in self._w_items:
            idx = self.gidx[off:off + w.numel()].long()
            out[key] = (g[idx] / self.loss_scale).view(w.shape)
        return out

    def state_dict(self) -> Dict[str, Tensor]:
        out = {key: self.w_flat[off:off + w.numel()].view(w.shape).clone() for key, w, off in self._w_items}
        for k, v in self.running_var.items():
            out[k + ".running_var"] = v.clone()
        return out

    def num_train_launches(self) -> int:
        return len(self.fwd_ops) + len(self.bwd_ops) + len(self.opt_ops) + 1

    def train_flops(self) -> float:
        """2*MAC of forward + data gradient + weight gradient (the data gradient of the stem is not needed)."""
        f = sum(l.fwd.algo_flops for l in self.layers)
        return 3.0 * f - self.stem.fwd.algo_flops


class ResNetTrainPlan(TrainPlanBase):
    """One fine-tuning step of `BcosifyNetwork(ResNetBcos(...))` on `batch` images per rank."""

    def __init__(self, arch: str, state_dict: Dict[str, Tensor], batch: int, **kw):
        self.kind, self.nblocks = RESNET_ARCH[arch]
        super().__init__(arch, state_dict, batch, **kw)

    def _build(self) -> None:
        sd = self.sd
        self.pool_out = self._stem("model.conv1.linear.weight", "model.bn1", pool_sq=True)
        x = self.pool_out
        self.blocks: List[dict] = []
        for li, (width, nblocks) in enumerate(zip([64, 128, 256, 512], self.nblocks), start=1):
            for bi in range(nblocks):
                stride = 2 if (li > 1 and bi == 0) else 1
                pfx = f"model.layer{li}.{bi}"
                ds = None
                idn = x.t
                if (pfx + ".downsample.0.linear.weight") in sd:
                    ds = self._conv_bn(pfx + ".downsample", x, pfx + ".downsample.0.linear.weight", stride, 0, pfx + ".downsample.1", False,
                                       want_z_sq=False)
                    idn = ds.z.t
                if self.kind == "basic":
                    c1 = self._conv_bn(pfx + ".conv1", x, pfx + ".conv1.linear.weight", stride, 1, pfx + ".bn1", True)
                    c2 = self._conv_bn(pfx + ".conv2", c1.z, pfx + ".conv2.linear.weight", 1, 1, pfx + ".bn2", True, res=idn)
                    convs = [c1, c2]
                else:
                    c1 = self._conv_bn(pfx + ".conv1", x, pfx + ".conv1.linear.weight", 1, 0, pfx + ".bn1", True)
                    c2 = self._conv_bn(pfx + ".conv2", c1.z, pfx + ".conv2.linear.weight", stride, 1, pfx + ".bn2", True)
                    c3 = self._conv_bn(pfx + ".conv3", c2.z, pfx + ".conv3.linear.weight", 1, 0, pfx + ".bn3", True, res=idn)
                    convs = [c1, c2, c3]
                self.blocks.append(dict(name=pfx, convs=convs, ds=ds, x=x, y=convs[-1].z))
                x = convs[-1].z
        self._head("fc", x, "model.fc.linear.weight")
        self._alloc_master()
        self._build_backward()
        if self.device.type == "cuda":
            self.refresh_operands()

    def _build_backward(self) -> None:
        # gradient buffer in BACKWARD order: classifier first, stem last, so that finished buckets are contiguous
        order = [self.fc]
        for blk in reversed(self.blocks):
            order += list(reversed(blk["convs"]))
            if blk["ds"] is not None:
                order.append(blk["ds"])
        order.append(self.stem)
        self._alloc_grads(order)
        # ---- classifier
        self._layer_bwd(self.fc, self.g_fc, None, None)
        ga, gb = self.fc.gx.view(-1, self.fc.rec.cin_phys), None
        tn = self.fc.gnT                                # 1x1 stride 1: the patch-norm vector is gnT itself
        # ---- blocks in reverse
        for bi in range(len(self.blocks) - 1, -1, -1):
            blk = self.blocks[bi]
            convs, ds = blk["convs"], blk["ds"]
            last = convs[-1]
            gy = self._layer_bwd(last, ga, gb, tn, want_gy=True)          # g_y also flows into the identity / downsample branch
            for j in range(len(convs) - 2, -1, -1):
                nxt, cur = convs[j + 1], convs[j]
                t_in = self._norm_vec(nxt)
                self._layer_bwd(cur, nxt.gx.view(-1, nxt.rec.cin_phys), None, t_in)
            first = convs[0]
            t_blk = self._norm_vec(first)
            if ds is not None:
                self._layer_bwd(ds, gy, None, None)
                self._norm_path(ds, t_blk, accumulate=True)
                gb = ds.gx.view(-1, ds.rec.cin_phys)
            else:
                gb = gy
            ga, tn = first.gx.view(-1, first.rec.cin_phys), t_blk
        # ---- pooled stem: g = ga + gb + x_pool * T, average-pool backward, stem layer
        M_pool = self.pool_out.t.shape[0] * self.pool_out.t.shape[1] * self.pool_out.t.shape[2]
        g_pool = self._empty(*self.pool_out.t.shape)
        self.bwd_ops.append(FnOp("pool.grad", lambda: L.grad_combine(ga, gb, self.pool_out.t, tn, M_pool, 64, g_pool, self.dt_code)))
        g_stem = self._empty(*self.stem.z.t.shape)
        self.bwd_ops.append(O.AvgPoolBwdMulOp("pool.bwd", g_pool, 64, 1, 3, 2, 1, None, g_stem, self.dt_code))
        self._layer_bwd(self.stem, g_stem.view(-1, 64), None, None)
        self._close_bucket()
        self._build_optimizer()


@dataclass
class DenseNorm:
    """A consumer's batch-statistics BN + ReLU over the prefix F[:, :c] of a dense block's feature tensor (dense-layer norm1, a
    transition's norm, norm5).  Its statistics are the block's per-channel ones; it owns alpha, its running_var and its BN weight."""
    name: str
    blk: "DenseTrainBlock"
    c: int
    t: Act                                   # relu(F[:, :c] * alpha), the input of the 1x1 conv that follows
    alpha: Tensor
    bnw_off: int
    gbn_off: int = -1
    conv: Optional[TrainLayer] = None        # the 1x1 B-cos conv that reads t (its gnT is the patch-norm path of t)


@dataclass
class DenseTrainBlock:
    name: str
    F: Tensor                                # [nb, h, w, c_total] 16-bit feature tensor
    c_total: int
    c_in: int
    M: int
    mean: Tensor                             # [c_total] fp32 batch statistics of every channel of F
    var: Tensor
    rstd: Tensor
    K: Tensor                                # [c_total] fp32: sum over the consumers of their batch-statistics coefficients k_l
    G: Tensor                                # [M, c_total] fp32 gradient wrt F (the consumers' direct terms)
    layers: List[Tuple[DenseNorm, TrainLayer, TrainLayer]] = field(default_factory=list)     # (norm1, conv1, conv2)
    t_norm: Optional[DenseNorm] = None       # transition behind the block
    t_conv: Optional[TrainLayer] = None


class DenseNetTrainPlan(TrainPlanBase):
    """One fine-tuning step of `BcosifyNetwork(DenseNetBcos(...))` (DenseNet-121 / -169 / -201) on `batch` images per rank.

    Same launches as the ResNet plan for the stem, the convs (+ norm2 of every dense layer) and the head.  What is DenseNet's own is
    the batch-statistics BN + ReLU every consumer applies to a prefix of its block's feature tensor F (csrc/bcosk_dense_train.cu):
      forward   dense_slice_stats after the block-input copy and after every 3x3 launch (statistics of a channel do not depend on the
                consumer: computed once), then per consumer dense_consumer_finalize -> dense_bn_relu_fwd -> its 1x1 conv
      backward  per consumer ONE pass dense_consumer_bwd (G[:, :C_l] += g_y alpha_l, S_l) + finalize (BN weight gradient, K += k_l);
                the batch-statistics terms of all consumers, (F - mean) K, are applied once by dense_slice_bwd when the slice's
                producer (a 3x3 conv, or the block input) runs its backward."""

    def __init__(self, arch: str, state_dict: Dict[str, Tensor], batch: int, **kw):
        from .densenet import DENSENET_ARCH
        self.growth, self.block_cfg, self.init_c = DENSENET_ARCH[arch]
        super().__init__(arch, state_dict, batch, **kw)

    # ------------------------------------------------------------------ forward
    def _slice_stats(self, blk: DenseTrainBlock, col0: int, c: int, name: str) -> None:
        part = self.stat_part[:self.red_blocks * 2 * c].view(self.red_blocks, 2 * c)
        self.fwd_ops.append(FnOp(name, lambda: L.dense_slice_stats(blk.F, blk.M, blk.c_total, col0, c, self.bn_eps, part, blk.mean, blk.var,
                                                                    blk.rstd, self.dt_code)))

    def _consumer(self, bn: str, blk: DenseTrainBlock, c: int) -> DenseNorm:
        nb = self.nb
        h, w = blk.F.shape[1], blk.F.shape[2]
        alpha = self._empty(c, dtype=torch.float32)
        off = self._cur_w_off
        self._w_items.append((bn + ".weight", self.sd[bn + ".weight"], off))
        self._cur_w_off += c
        rv = self._dev(self.sd[bn + ".running_var"])
        self.running_var[bn] = rv
        self.fwd_ops.append(FnOp(bn + ".finalize", lambda: L.dense_consumer_finalize(blk.var, blk.rstd, self.w_flat[off:off + c], c, self.momentum,
                                                                                     rv, alpha)))
        t = self._empty(nb, h, w, c)
        sq = self._empty(1, nb * h * w, dtype=torch.float32)
        self.fwd_ops.append(O.DenseBnReluFwdOp(bn + ".apply", blk.F, c, 1, alpha, True, t, sq, None, self.dt_code))
        return DenseNorm(bn, blk, c, Act(t, c, sq, 1), alpha, off)

    def _build(self) -> None:
        from .densenet import dn_names
        nb = self.nb
        nm = dn_names(len(self.block_cfg))
        f32 = dict(dtype=torch.float32)
        pooled = self._stem(nm["conv0"] + ".linear.weight", nm["norm0"], pool_sq=False).t
        hw = (pooled.shape[1], pooled.shape[2])
        c = self.init_c
        # per-block partial sums, shared by the launches (one stream): statistics [blocks][2 c], consumer reductions [blocks][c]
        c_max = max(ci + self.growth * n for ci, n in zip(self._block_inputs(), self.block_cfg))
        self.stat_part = self._empty(self.red_blocks * 2 * c_max, **f32)
        self.cons_part = self._empty(self.red_blocks * c_max, **f32)
        self.blocks: List[DenseTrainBlock] = []
        self.norms: List[DenseNorm] = []
        for bi, nlayers in enumerate(self.block_cfg, start=1):
            c_total = c + self.growth * nlayers
            M = nb * hw[0] * hw[1]
            F = self._zeros(nb, hw[0], hw[1], c_total)
            blk = DenseTrainBlock(f"denseblock{bi}", F, c_total, c, M, *(self._zeros(c_total, **f32) for _ in range(4)),
                                  G=self._empty(M, c_total, **f32))
            self.blocks.append(blk)
            self.fwd_ops.append(O.CopyChannelsOp(f"denseblock{bi}.input", pooled, c, 1, F, 0))
            self._slice_stats(blk, 0, c, f"denseblock{bi}.input.stats")
            cl = c
            for li in range(1, nlayers + 1):
                p = nm[f"denseblock{bi}"] + f".denselayer{li}"
                n1 = self._consumer(p + ".norm1", blk, cl)
                c1 = self._conv_bn(p + ".conv1", n1.t, p + ".conv1.linear.weight", 1, 0, p + ".norm2", True)
                n1.conv = c1
                c2 = self._conv_bn(p + ".conv2", c1.z, p + ".conv2.linear.weight", 1, 1, None, False, y_buf=F, y_col=cl)
                self._slice_stats(blk, cl, self.growth, p + ".conv2.stats")
                blk.layers.append((n1, c1, c2))
                self.norms.append(n1)
                cl += self.growth
            c = c_total
            if bi != len(self.block_cfg):
                tn = self._consumer(nm[f"transition{bi}.norm"], blk, c)
                tc = self._conv_bn(nm[f"transition{bi}.conv"], tn.t, nm[f"transition{bi}.conv"] + ".linear.weight", 1, 0, None, False)
                tn.conv = tc
                blk.t_norm, blk.t_conv = tn, tc
                self.norms.append(tn)
                c //= 2
                y = tc.out.view(nb, hw[0], hw[1], c)
                hw = (hw[0] // 2, hw[1] // 2)
                pooled = self._empty(nb, hw[0], hw[1], c)
                self.fwd_ops.append(O.AvgPoolFwdOp(f"transition{bi}.pool", y, c, 1, 2, 2, 0, pooled, self.dt_code, None))
        n5 = self._consumer(nm["norm5"], self.blocks[-1], c)
        self.norms.append(n5)
        self.norm5 = n5
        self._head("classifier", n5.t, "model.classifier.linear.weight")
        n5.conv = self.fc
        self._alloc_master()
        self._build_backward()
        if self.device.type == "cuda":
            self.refresh_operands()

    def _block_inputs(self) -> List[int]:
        c, out = self.init_c, []
        for bi, n in enumerate(self.block_cfg):
            out.append(c)
            c = (c + self.growth * n) // 2
        return out

    # ------------------------------------------------------------------ backward
    def _consumer_bwd(self, n: DenseNorm, accumulate: bool) -> None:
        """g_t (the consumer conv's fp32 data gradient) -> G[:, :c] and the partials of S, then the BN weight gradient and K += k."""
        blk, c, M, dtc = n.blk, n.c, n.blk.M, self.dt_code
        g_t = n.conv.gx.view(M, c)
        part = self.cons_part[:self.red_blocks * c].view(self.red_blocks, c)
        self.bwd_ops.append(FnOp(n.name + ".bwd", lambda: L.dense_consumer_bwd(g_t, n.t.t, n.conv.gnT, n.alpha, blk.F, blk.c_total, M, c, blk.G,
                                                                             accumulate, part, dtc)))
        self.bwd_ops.append(FnOp(n.name + ".bwd.finalize", lambda: L.dense_consumer_bwd_finalize(
            part, blk.rstd, self.w_flat[n.bnw_off:n.bnw_off + c], M, c, accumulate, blk.K, self.g_flat[n.gbn_off:n.gbn_off + c])))
        self._grad_ready_to(n.gbn_off + c)

    def _consumer_conv_bwd(self, lay: TrainLayer, ga: Tensor, n: DenseNorm, scratch: Tensor, accumulate: bool) -> None:
        """A consumer's 1x1 conv without a norm behind it (transition, classifier): B-cos backward, weight gradient, fp32 data
        gradient into `scratch`, then the consumer's own backward."""
        self._layer_bwd(lay, ga, None, None, gx32=scratch[:n.blk.M * n.c].view(self.nb, *n.t.hw, n.c))
        self._consumer_bwd(n, accumulate)

    def _build_backward(self) -> None:
        nb, dtc = self.nb, self.dt_code
        order: List = [self.fc, self.norm5]
        for blk in reversed(self.blocks):
            for n1, c1, c2 in reversed(blk.layers):
                order += [c2, c1, n1]
            prev = self.blocks.index(blk) - 1
            if prev >= 0:
                order += [self.blocks[prev].t_conv, self.blocks[prev].t_norm]
        order.append(self.stem)
        self._alloc_grads(order)
        self.norm_units = [(n.bnw_off, n.gbn_off, n.c) for n in self.norms]
        scratch = self._empty(max(b.M * b.c_total for b in self.blocks), dtype=torch.float32)   # fp32 data gradients of the 1x1 convs
        # ---- head: classifier, then norm5 (the first consumer of the last block: it writes G and K)
        self._consumer_conv_bwd(self.fc, self.g_fc, self.norm5, scratch, accumulate=False)
        for bi in range(len(self.blocks) - 1, -1, -1):
            blk = self.blocks[bi]
            M = blk.M
            for n1, c1, c2 in reversed(blk.layers):
                # 3x3 slice: g_out = G + (F - mean) K -> g_lin, gnT; weight and data gradient
                self._alloc_ghat(c2.rec, classes=True)
                glin = c2.rec.ghat.view(M, self.growth)
                col = n1.c
                self.bwd_ops.append(FnOp(c2.name + ".bwd.slice", lambda blk=blk, c2=c2, glin=glin, col=col: L.dense_slice_bwd(
                    blk.G, blk.F, blk.c_total, col, blk.M, self.growth, blk.mean, blk.K, c2.rec.gain, c2.rec.inv, glin, c2.gnT, dtc)))
                self._wgrad_dgrad(c2, glin)
                # conv1 + norm2 (+ ReLU) with the 3x3's patch-norm path, its data gradient in fp32, then norm1's one pass
                self._layer_bwd(c1, c2.gx.view(-1, c2.rec.cin_phys), None, self._norm_vec(c2),
                                gx32=scratch[:M * n1.c].view(nb, *n1.t.hw, n1.c))
                self._consumer_bwd(n1, accumulate=True)
            # ---- the block's input channels: g = G[:, :c_in] + (F - mean) K, through the pool in front of the block
            g_in = self._empty(nb, *blk.F.shape[1:3], blk.c_in)
            self.bwd_ops.append(FnOp(blk.name + ".input.bwd", lambda blk=blk, g_in=g_in: L.dense_slice_bwd(
                blk.G, blk.F, blk.c_total, 0, blk.M, blk.c_in, blk.mean, blk.K, None, None, g_in, None, dtc)))
            if bi > 0:
                prev = self.blocks[bi - 1]
                tc = prev.t_conv
                g_y = self._empty(*tc.out.shape)
                h, w = prev.F.shape[1], prev.F.shape[2]
                self.bwd_ops.append(O.AvgPoolBwdMulOp(f"transition{bi}.pool.bwd", g_in, blk.c_in, 1, 2, 2, 0, None, g_y.view(nb, h, w, blk.c_in),
                                                      dtc))
                self._consumer_conv_bwd(tc, g_y, prev.t_norm, scratch, accumulate=False)
            else:
                g_stem = self._empty(*self.stem.z.t.shape)
                self.bwd_ops.append(O.AvgPoolBwdMulOp("pool.bwd", g_in, blk.c_in, 1, 3, 2, 1, None, g_stem, dtc))
                self._layer_bwd(self.stem, g_stem.view(-1, blk.c_in), None, None)
        self._close_bucket()
        self._build_optimizer()
