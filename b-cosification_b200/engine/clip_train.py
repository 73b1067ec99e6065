"""Fine-tuning step of the B-cosified CLIP ResNet image encoder (the reference's CLIP configs, bcos/training with `clip_kd`): forward
in train mode to the [batch, D] embedding, the user's loss on that embedding in torch, the full backward (trunk and attention-pool
head, q and k in the graph), the bucketed gradient all-reduce, AGC + AdamW and the operand refresh.

Network: CLIP/clip/model.py:94-154 `ModifiedResNet` (three-conv stem + AvgPool2d(2); model.py:10-55 `Bottleneck` with the stride
in an AvgPool2d after conv2 and in front of the downsample conv) and `BcosAttentionPool2d` (bcos/modules/bcosattnpool.py:34-59),
as in engine/clip_rn.py and `OracleCLIPResNet`.

Trunk: the conv + batch-statistics BN launches and their backward are TrainPlanBase's.  The 3x3/2 stem conv runs as a 2x2/1 conv
over the space-to-depth input; its stand-in goes through `stem_s2d_weight`, so its packed elements point back at the 3x3 master
weights.  Every average pool's backward is ONE pass (`bcosk_pool_bwd_norm`) that also applies the consumers' terms at the pooled
resolution (their data gradients and the patch-norm path x * T).

Head (fp32, commuted as in the inference plan: no projection of the 50 tokens).  Per image and head h, with x_j the tokens
(x_0 = mean token), q = W_q x_0 / sqrt(dh), q~_h = W_k,h^T q_h, s_j = q~_h . x_j, p = softmax(s), xbar_h = sum_j p_j x_j,
o_h = W_v,h xbar_h, emb = W_c o, the backward of g_emb is
    dW_c = g_emb^T o                 g_o = W_c^T g_emb
    dW_v,h = g_o,h^T xbar_h          g_xbar_h = W_v,h^T g_o,h
    dp_j = g_xbar_h . x_j            ds = p (dp - sum_j p_j dp_j)                    (bcosk_softmax_bwd)
    g_q~_h = sum_j ds_j x_j          dW_k,h = q_h^T g_q~_h      g_q,h = W_k,h g_q~_h      dW_q = g_q^T x_0 / sqrt(dh)
    g_x_j = sum_h p_j g_xbar_h + sum_h ds_j q~_h  (+ W_q^T g_q / sqrt(dh) for j = 0)
and `bcosk_seed_from_tokens` spreads the mean token's share over the pixels.  All of it is `bcosk_sgemm_batched` over the fp32 master
weights (nothing to refresh); the gradients land in the flat buffer, one AGC unit per output row.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Callable, Dict, List, Optional

import torch
from torch import Tensor

from .. import _lib as L
from . import ops as O
from . import pack as P
from .base import Act
from .clip_rn import CLIP_MEAN_ADDINVERSE, CLIP_STD_ADDINVERSE
from .train import FnOp, TrainLayer, TrainPlanBase


@dataclass
class HeadWeight:
    """An fp32 head matrix [rows, cols] used unpacked by the SGEMM launches (a gradient slot of rows * cols, one AGC unit per row)."""
    key: str
    w_off: int
    rows: int
    cols: int
    gbn_off: int = -1            # its gradient slot (`_alloc_grads` fills it like a norm record's)

    @property
    def c(self) -> int:
        return self.rows * self.cols


@dataclass
class ClipTrainBlock:
    name: str
    convs: List[TrainLayer]
    ds: Optional[TrainLayer]
    stride: int
    t2p: Optional[Act]           # conv2's output after the block's pool (stride > 1)
    xp: Optional[Act]            # the block input after the downsample's pool (stride > 1)


class CLIPResNetTrainPlan(TrainPlanBase):
    """One fine-tuning step of the B-cosified CLIP ResNet image encoder on `batch` images per rank.  The loss is a function of the
    embedding: `train_step(images, loss_fn)`.  Only b = 2 is built."""

    def __init__(self, state_dict: Dict[str, Tensor], batch: int, *, layers=(3, 4, 6, 3), width: int = 64, heads: int = 32,
                 b: float = 2.0, mean=CLIP_MEAN_ADDINVERSE, std=CLIP_STD_ADDINVERSE, **kw):
        if float(b) != 2.0:
            raise ValueError(f"CLIPResNetTrainPlan: only b = 2 is built (got b = {b})")
        self.stage_cfg, self.width, self.heads = tuple(layers), width, heads
        self._graphs = None
        self.last_loss: Optional[Tensor] = None
        super().__init__("clip_rn", state_dict, batch, mean=mean, std=std, logit_bias=None, **kw)

    # ------------------------------------------------------------------ forward
    def _pool(self, name: str, x: Act, s: int) -> Act:
        h, w = x.hw
        y = self._empty(self.nb, h // s, w // s, x.c)
        sq = self._empty(1, self.nb * (h // s) * (w // s), dtype=torch.float32)
        self.fwd_ops.append(O.AvgPoolFwdOp(name, x.t, x.c, 1, s, s, 0, y, self.dt_code, sq))
        return Act(y, x.c, sq, 1)

    def _build(self) -> None:
        nb, S, sd, cp = self.nb, self.size, self.sd, 32
        if S % 32:
            raise ValueError("CLIP ResNets reduce the resolution 32x: image_size must be a multiple of 32")
        self.x_in = self._empty(nb, 3, S, S, dtype=torch.uint8) if self.input_u8 else self._empty(nb, 6, S, S, dtype=torch.float32)
        h2 = S // 2
        a0 = self._empty(nb, h2, h2, cp)
        sq0 = self._empty(1, nb * S * S, dtype=torch.float32)
        self.fwd_ops.append(O.InputPrepOp("input_prep", self.x_in, self.mean, self.inv_std, a0, cp, 1, self.dt_code, sq0))
        # stem: 3x3/2 as 2x2/1 over the space-to-depth input (patch norm = the original 3x3/2 pad-1 window), 3x3, 3x3, avg pool 2
        w3, off3 = self._register_weight("model.conv1.linear.weight")
        s1 = self._conv_bn("stem.conv1", Act(a0, cp, sq0, 1), "", 1, 1, "model.bn1", True, w_standin=P.stem_s2d_weight(w3, cp), w_off=off3,
                           w_numel=w3.numel(), pad_hi=0, kch=32, sq_geom=(S, S, 3, 2, 1))
        s1.need_dgrad = False
        s2 = self._conv_bn("stem.conv2", s1.z, "model.conv2.linear.weight", 1, 1, "model.bn2", True, kch=32)
        s3 = self._conv_bn("stem.conv3", s2.z, "model.conv3.linear.weight", 1, 1, "model.bn3", True, kch=32, want_z_sq=False)
        self.stem, self.stem_convs = s1, [s1, s2, s3]
        x = self.pool_out = self._pool("stem.pool", s3.z, 2)
        self.blocks: List[ClipTrainBlock] = []
        for li, nblocks in enumerate(self.stage_cfg, start=1):
            for bi in range(nblocks):
                s = 2 if (li > 1 and bi == 0) else 1
                pfx = f"model.layer{li}.{bi}"
                c1 = self._conv_bn(pfx + ".conv1", x, pfx + ".conv1.linear.weight", 1, 0, pfx + ".bn1", True)
                c2 = self._conv_bn(pfx + ".conv2", c1.z, pfx + ".conv2.linear.weight", 1, 1, pfx + ".bn2", True, want_z_sq=s == 1)
                t2p = self._pool(pfx + ".avgpool", c2.z, s) if s > 1 else None
                ds, xp, idn = None, None, x.t
                if (pfx + ".downsample.1.linear.weight") in sd:
                    xp = self._pool(pfx + ".downsample.0", x, s) if s > 1 else None
                    ds = self._conv_bn(pfx + ".downsample", x if xp is None else xp, pfx + ".downsample.1.linear.weight", 1, 0, pfx + ".downsample.2", False,
                                       want_z_sq=False)
                    idn = ds.z.t
                c3 = self._conv_bn(pfx + ".conv3", c2.z if t2p is None else t2p, pfx + ".conv3.linear.weight", 1, 0, pfx + ".bn3", True, res=idn)
                self.blocks.append(ClipTrainBlock(pfx, [c1, c2, c3], ds, s, t2p, xp))
                x = c3.z
        self.trunk_out = x
        # head weights: fp32 masters read by the SGEMM launches directly
        C = x.c
        self.head_w: Dict[str, HeadWeight] = {}
        for nme in ("q_proj", "k_proj", "v_proj", "c_proj"):
            key = f"model.attnpool.{nme}.weight" if nme != "c_proj" else "model.attnpool.c_proj.linear.weight"
            _, off = self._register_weight(key)
            rows, cols = self.sd[key].shape
            assert cols == C, (key, cols, C)
            self.head_w[nme] = HeadWeight(key, off, rows, cols)
        self._alloc_master()
        self._build_head_forward()
        self._build_backward()
        if self.device.type == "cuda":
            self.refresh_operands()

    def _hw(self, nme: str, grad: bool = False) -> Tensor:
        hw = self.head_w[nme]
        buf, off = (self.g_flat, hw.gbn_off) if grad else (self.w_flat, hw.w_off)
        return buf[off:off + hw.c].view(hw.rows, hw.cols)

    def _build_head_forward(self) -> None:
        nb, H = self.nb, self.heads
        C = self.trunk_out.c
        dh = C // H
        T = self.trunk_out.hw[0] * self.trunk_out.hw[1] + 1
        f32 = torch.float32
        wq, wk, wv, wc = (self._hw(n) for n in ("q_proj", "k_proj", "v_proj", "c_proj"))
        od = wc.shape[0]
        self.tokens = self._empty(nb, T, C, dtype=f32)
        self.h_q = self._empty(nb, C, dtype=f32)
        self.h_qt = self._empty(nb, H, C, dtype=f32)
        self.h_p = self._empty(nb, H, T, dtype=f32)
        self.h_xbar = self._empty(nb, H, C, dtype=f32)
        self.h_o = self._empty(nb, C, dtype=f32)
        self.emb = self._empty(nb, od, dtype=f32)
        self.q_scale = dh ** -0.5
        ops = self.fwd_ops
        ops.append(O.HeadTokensOp("attnpool.tokens", self.trunk_out.t, C, 1, self.dt_code, self.tokens))
        ops.append(O.SgemmOp("attnpool.q", False, True, nb, C, C, self.tokens, 0, T * C, 0, wq, 0, C, 0, self.h_q, 0, C, 0, 1, self.q_scale))
        ops.append(O.SgemmOp("attnpool.qk", False, False, nb, C, dh, self.h_q, 0, C, dh, wk, 0, C, dh * C, self.h_qt, 0, H * C, C, H))
        ops.append(O.SgemmOp("attnpool.scores", False, True, H, T, C, self.h_qt, 0, C, H * C, self.tokens, 0, C, T * C, self.h_p, 0, T, H * T, nb))
        ops.append(O.RowSoftmaxOp("attnpool.softmax", self.h_p))
        ops.append(O.SgemmOp("attnpool.pool", False, False, H, C, T, self.h_p, 0, T, H * T, self.tokens, 0, C, T * C, self.h_xbar, 0, C, H * C, nb))
        ops.append(O.SgemmOp("attnpool.v", False, True, nb, dh, C, self.h_xbar, 0, H * C, C, wv, 0, C, dh * C, self.h_o, 0, C, dh, H))
        ops.append(O.SgemmOp("attnpool.c_proj", False, True, nb, od, C, self.h_o, 0, C, 0, wc, 0, C, 0, self.emb, 0, od, 0, 1))

    # ------------------------------------------------------------------ backward
    def _pool_bwd(self, name: str, ga: Tensor, gb: Optional[Tensor], xp: Act, tn: Optional[Tensor], gx: Tensor, k: int) -> None:
        """gx = AvgPool2d(k) backward of (ga + gb + xp * tn) (the pooled tensor's consumers' terms), one pass."""
        nb, h, w, c = gx.shape
        self.bwd_ops.append(FnOp(name, lambda: L.pool_bwd_norm(ga, False, gb, xp.t, tn, nb, h, w, c, k, False, gx, self.dt_code)))

    def _build_head_backward(self) -> Tensor:
        """Head backward (module docstring); returns the 16-bit gradient wrt the trunk output."""
        nb, H = self.nb, self.heads
        C = self.trunk_out.c
        dh, T = C // H, self.tokens.shape[1]
        f32 = torch.float32
        wq, wk, wv, wc = (self._hw(n) for n in ("q_proj", "k_proj", "v_proj", "c_proj"))
        gq_w, gk_w, gv_w, gc_w = (self._hw(n, grad=True) for n in ("q_proj", "k_proj", "v_proj", "c_proj"))
        od = wc.shape[0]
        self.g_emb = self._zeros(nb, od, dtype=f32)
        self.g_o = self._empty(nb, C, dtype=f32)
        self.g_xbar = self._empty(nb, H, C, dtype=f32)
        self.g_s = self._empty(nb, H, T, dtype=f32)          # d loss / d p, then (in place) d loss / d scores
        self.g_qt = self._empty(nb, H, C, dtype=f32)
        self.g_q = self._empty(nb, C, dtype=f32)
        self.g_tokens = self._empty(nb, T, C, dtype=f32)
        ops, s = self.bwd_ops, self.q_scale
        ops.append(O.SgemmOp("attnpool.c_proj.wgrad", True, False, od, C, nb, self.g_emb, 0, od, 0, self.h_o, 0, C, 0, gc_w, 0, C, 0, 1))
        ops.append(O.SgemmOp("attnpool.c_proj.bwd", False, False, nb, C, od, self.g_emb, 0, od, 0, wc, 0, C, 0, self.g_o, 0, C, 0, 1))
        ops.append(O.SgemmOp("attnpool.v.wgrad", True, False, dh, C, nb, self.g_o, 0, C, dh, self.h_xbar, 0, H * C, C, gv_w, 0, C, dh * C, H))
        ops.append(O.SgemmOp("attnpool.v.bwd", False, False, nb, C, dh, self.g_o, 0, C, dh, wv, 0, C, dh * C, self.g_xbar, 0, H * C, C, H))
        ops.append(O.SgemmOp("attnpool.p.bwd", False, True, H, T, C, self.g_xbar, 0, C, H * C, self.tokens, 0, C, T * C, self.g_s, 0, T, H * T, nb))
        ops.append(FnOp("attnpool.softmax.bwd", lambda: L.softmax_bwd(self.h_p, self.g_s, nb * H, T, self.g_s)))
        ops.append(O.SgemmOp("attnpool.qk.bwd", False, False, H, C, T, self.g_s, 0, T, H * T, self.tokens, 0, C, T * C, self.g_qt, 0, C, H * C, nb))
        ops.append(O.SgemmOp("attnpool.k.wgrad", True, False, dh, C, nb, self.h_q, 0, C, dh, self.g_qt, 0, H * C, C, gk_w, 0, C, dh * C, H))
        ops.append(O.SgemmOp("attnpool.q.bwd", False, True, nb, dh, C, self.g_qt, 0, H * C, C, wk, 0, C, dh * C, self.g_q, 0, C, dh, H))
        ops.append(O.SgemmOp("attnpool.q.wgrad", True, False, C, C, nb, self.g_q, 0, C, 0, self.tokens, 0, T * C, 0, gq_w, 0, C, 0, 1, s))
        # token gradient: values / pooling path, scores path (keys), query path into the mean token
        ops.append(O.SgemmOp("attnpool.tokens.bwd.v", True, False, T, C, H, self.h_p, 0, T, H * T, self.g_xbar, 0, C, H * C, self.g_tokens, 0, C,
                             T * C, nb))
        ops.append(O.SgemmOp("attnpool.tokens.bwd.k", True, False, T, C, H, self.g_s, 0, T, H * T, self.h_qt, 0, C, H * C, self.g_tokens, 0, C,
                             T * C, nb, accumulate=True))
        ops.append(O.SgemmOp("attnpool.tokens.bwd.q", False, False, nb, C, C, self.g_q, 0, C, 0, wq, 0, C, 0, self.g_tokens, 0, T * C, 0, 1, s,
                             accumulate=True))
        self._grad_ready_to(max(hw.gbn_off + hw.c for hw in self.head_w.values()))
        g_trunk = self._empty(*self.trunk_out.t.shape)
        ops.append(O.SeedFromTokensOp("attnpool.seed", self.g_tokens, 1.0, None, g_trunk, None, None, None, 1, self.dt_code))
        return g_trunk

    def _build_backward(self) -> None:
        # gradient buffer in backward order: the head first (c_proj, v, k, q), the stem last
        order: List = [self.head_w[n] for n in ("c_proj", "v_proj", "k_proj", "q_proj")]
        for blk in reversed(self.blocks):
            order += list(reversed(blk.convs))
            if blk.ds is not None:
                order.append(blk.ds)
        order += list(reversed(self.stem_convs))
        self._alloc_grads(order)
        self.row_units = [(hw.w_off, hw.gbn_off, hw.rows, hw.cols) for hw in order[:4]]
        ga, gb, tn = self._build_head_backward(), None, None
        ga = ga.view(-1, self.trunk_out.c)
        for blk in reversed(self.blocks):
            c1, c2, c3 = blk.convs
            gy = self._layer_bwd(c3, ga, gb, tn, want_gy=True)        # g_y also flows into the identity / downsample branch
            if blk.stride > 1:
                # conv2's output reaches conv3 through the block's pool: its gradient is the pool's backward of conv3's terms
                g_z2 = self._empty(*c2.z.t.shape)
                self._pool_bwd(blk.name + ".avgpool.bwd", c3.gx.view(-1, c3.rec.cin_phys), None, blk.t2p, c3.gnT, g_z2, blk.stride)
                self._layer_bwd(c2, g_z2.view(-1, c2.fwd.n), None, None)
            else:
                self._layer_bwd(c2, c3.gx.view(-1, c3.rec.cin_phys), None, self._norm_vec(c3))
            self._layer_bwd(c1, c2.gx.view(-1, c2.rec.cin_phys), None, self._norm_vec(c2))
            tn = c1.gnT                                                # 1x1 stride 1: the patch-norm vector of the block input
            if blk.ds is None:
                gb = gy
            elif blk.stride > 1:
                self._layer_bwd(blk.ds, gy, None, None)
                gb = self._empty(self.nb, *c1.rec.in_hw, c1.rec.cin_phys)
                self._pool_bwd(blk.name + ".downsample.0.bwd", blk.ds.gx.view(-1, blk.ds.rec.cin_phys), None, blk.xp, blk.ds.gnT, gb, blk.stride)
                gb = gb.view(-1, c1.rec.cin_phys)
            else:
                self._layer_bwd(blk.ds, gy, None, None)
                self._norm_path(blk.ds, tn, accumulate=True)
                gb = blk.ds.gx.view(-1, blk.ds.rec.cin_phys)
            ga = c1.gx.view(-1, c1.rec.cin_phys)
        # ---- stem: pool backward of the first block's terms, three conv layers (conv1 needs no data gradient)
        s1, s2, s3 = self.stem_convs
        g_z3 = self._empty(*s3.z.t.shape)
        self._pool_bwd("stem.pool.bwd", ga, gb, self.pool_out, tn, g_z3, 2)
        self._layer_bwd(s3, g_z3.view(-1, s3.fwd.n), None, None)
        self._layer_bwd(s2, s3.gx.view(-1, s3.rec.cin_phys), None, self._norm_vec(s3))
        self._layer_bwd(s1, s2.gx.view(-1, s2.rec.cin_phys), None, self._norm_vec(s2))
        self._close_bucket()
        self._build_optimizer()

    # ------------------------------------------------------------------ execution
    def _loss_grad(self, loss_fn: Callable[[Tensor], Tensor]) -> Tensor:
        """The user's loss on an fp32 leaf copy of the embedding; d loss / d emb (x loss_scale) goes into the head's gradient buffer."""
        emb = self.emb.detach().clone().requires_grad_(True)
        with torch.enable_grad():
            loss = loss_fn(emb)
            (g,) = torch.autograd.grad(loss * self.loss_scale, [emb])
        self.g_emb.copy_(g)
        return loss.detach()

    def _backward_step(self) -> None:
        O.run_ops(self.bwd_ops)
        if self.world > 1:
            torch.cuda.current_stream().wait_stream(self.comm_stream)
        O.run_ops(self.opt_ops)
        self.refresh_operands()

    def embed(self, images: Optional[Tensor] = None) -> Tensor:
        """Train-mode forward only (batch statistics; updates the BN running variances): the embedding [batch, D] fp32."""
        self._require_gpu()
        if images is not None:
            self.x_in.copy_(images, non_blocking=True)
        if self._graphs is not None:
            self._graphs[0].replay()
        else:
            O.run_ops(self.fwd_ops)
        return self.emb

    def forward_backward(self, loss_fn: Callable[[Tensor], Tensor]) -> Tensor:
        """Forward (train mode), `loss_fn(embedding)`, backward and the gradient all-reduce; no optimizer step.  Returns the loss."""
        self.embed()
        self.last_loss = self._loss_grad(loss_fn)
        O.run_ops(self.bwd_ops)
        if self.world > 1:
            torch.cuda.current_stream().wait_stream(self.comm_stream)
        return self.last_loss

    def train_step(self, images: Optional[Tensor], loss_fn: Callable[[Tensor], Tensor]) -> Tensor:
        """One step: forward (train mode) -> embedding; `loss_fn(embedding)` (a scalar, torch); backward, gradient all-reduce,
        AGC + AdamW, operand refresh.  `images`: uint8 [batch, 3, S, S] (input_u8) or the 6-channel fp32 input; None keeps the
        loaded batch.  Returns the loss."""
        if images is not None:
            self.x_in.copy_(images, non_blocking=True)
        if self._graphs is None:
            loss = self.forward_backward(loss_fn)
            self.optimizer_step()
            return loss
        self._graphs[0].replay()
        self.last_loss = self._loss_grad(loss_fn)
        self.step_count += 1
        self._graphs[1].replay()
        return self.last_loss

    def capture(self) -> bool:
        """Capture two CUDA graphs, the forward and backward + optimizer + refresh, around the user's loss (which runs eagerly in
        between).  The training state is restored after the warm-up step the capture needs.  Single-rank plans only: returns False
        (the step stays eager) when world_size > 1."""
        self._require_gpu()
        if self.world > 1:
            return False
        state = [self.w_flat, self.m_flat, self.v_flat, self.adam_state, self.g_emb] + list(self.running_var.values())
        keep = [t.clone() for t in state]

        def restore():
            for dst, src in zip(state, keep):
                dst.copy_(src)
            self.refresh_operands()

        side = torch.cuda.Stream(self.device)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            O.run_ops(self.fwd_ops)
            self._backward_step()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        restore()
        g_fwd, g_bwd = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        try:
            with torch.cuda.graph(g_fwd):
                O.run_ops(self.fwd_ops)
            with torch.cuda.graph(g_bwd):
                self._backward_step()
        except Exception as e:  # noqa: BLE001
            import warnings
            warnings.warn(f"bcos_b200: CLIP training step not captured ({type(e).__name__}: {e}); running eagerly")
            torch.cuda.synchronize()
            restore()
            return False
        torch.cuda.synchronize()
        restore()
        self._graphs = (g_fwd, g_bwd)
        return True

    def train_flops(self) -> float:
        """2*MAC of the trunk's forward + data gradient + weight gradient (no data gradient of stem conv1) and of the head."""
        nb, C, T = self.nb, self.trunk_out.c, self.tokens.shape[1]
        od = self.head_w["c_proj"].rows
        head_fwd = 2.0 * nb * (3 * C * C + 2 * self.heads * T * C + od * C)
        return super().train_flops() + 3.0 * head_fwd
