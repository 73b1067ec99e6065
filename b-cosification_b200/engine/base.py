"""Shared machinery of the fused execution plans: buffers, forward conv emission, explain-dgrad emission.

A plan owns its device buffers (NHWC 16-bit activations with optional precision planes, fp32 side
tensors) and two flat launch lists, `fwd_ops` and `bwd_ops` (engine/ops.py).  Concrete networks
(engine/resnet.py, ...) only decide which launches to emit.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

import torch
from torch import Tensor

from .. import _lib as L
from . import ops as O
from . import pack as P

@dataclass
class Act:
    """An activation tensor in HBM: [nb, h, w, planes*c] + partial per-pixel sums of squares."""
    t: Tensor
    c: int
    sq: Optional[Tensor] = None      # [parts, nb*h*w] fp32
    parts: int = 0

    @property
    def hw(self) -> Tuple[int, int]:
        return self.t.shape[1], self.t.shape[2]


@dataclass
class ConvRec:
    """What the explanation pass needs to remember about one fused conv launch."""
    name: str
    w: Tensor                 # [o, c, kh, kw] fp32 as seen by the GEMM (stem: space-to-depth form)
    stride: int
    pad_lo: int
    pad_hi: int
    in_hw: Tuple[int, int]
    out_hw: Tuple[int, int]
    cin_phys: int             # channels per plane of the input tensor
    gain: Optional[Tensor] = None
    mask: Optional[Tensor] = None
    ghat: Optional[Tensor] = None          # gradient wrt the pre-scale linear output (x gain), maybe zero-inserted
    ghat_map: Optional[Tuple[int, int, int, int]] = None
    algo_flops: float = 0.0
    # gain not stored (include/bcosk.h mul1_sqrt_scale): recomputed as sqrt(y * inv) from the ReLU output and 1/||patch||
    gain_y: Optional[Tensor] = None
    gain_inv: Optional[Tensor] = None
    inv: Optional[Tensor] = None           # [M] fp32 1/||patch|| the forward launch used (kept for the training backward)
    amax: Optional[Tensor] = None          # MaxOut: [M, cout / max_out] uint8 index of the kept unit of every group

    @property
    def k(self) -> int:
        return self.w.shape[2]

    @property
    def cout(self) -> int:
        return self.w.shape[0]


@dataclass
class BlockRec:
    name: str
    convs: List[ConvRec]
    ds: Optional[ConvRec]
    x: Act
    y: Act
    mask: Tensor
    side: Optional[Tensor] = None   # gradient entering the identity / downsample branch



class PlanBase:
    """Buffers + launch emission shared by all network plans."""

    def __init__(self, batch: int, *, planes: int = 1, dtype: str = "bf16", device="cuda", explain: bool = True,
                 b: float = 2.0, bn_eps: float = 1e-5, state_dict: Optional[Dict[str, Tensor]] = None,
                 explain_planes: Optional[int] = None):
        self.nb, self.planes, self.device = batch, planes, torch.device(device)
        # Precision planes of the explanation pass (gradients, their weights, the saved gains).  The forward pass of a
        # random-init deep B-cos net is chaotic (a rounding error flips ReLU masks and moves every gain downstream), the
        # explanation pass is LINEAR in the gradient once gains and masks are fixed: rounding g, W and the gains to one
        # fp16 plane there costs 2-4e-4 of the map range (measured against the reference golden, DESIGN.md section 4),
        # so `planes=2, explain_planes=1` meets the parity contract at close to the one-plane cost for half of the step.
        self.bplanes = planes if explain_planes is None else int(explain_planes)
        assert 1 <= self.bplanes <= planes
        self.dt_code = L.DTYPE_CODE[dtype]
        self.dt = torch.bfloat16 if dtype == "bf16" else torch.float16
        self.gain_dt = self.dt if self.bplanes == 1 else torch.float32
        self.hp_accum = planes > 1        # parity mode: fp32-faithful accumulation (see include/bcosk.h hp_accum)
        self.bwd_hp = self.bplanes > 1
        self.b, self.bn_eps = float(b), bn_eps
        self.scale_mode = L.BCOSK_SCALE_NONE if b == 1 else (L.BCOSK_SCALE_B2 if b == 2 else L.BCOSK_SCALE_POW)
        self.sd = {k: v.detach().to(torch.float32) for k, v in (state_dict or {}).items() if v.is_floating_point()}
        self.with_explain = explain
        self.fwd_ops: List = []
        self.bwd_ops: List = []
        self._graph_fwd = None
        self._graph_all = None
        self._graph_bwd = None

    # ------------------------------------------------------------------ allocation helpers
    def _zeros(self, *shape, dtype=None) -> Tensor:
        return torch.zeros(*shape, dtype=dtype or self.dt, device=self.device)

    def _empty(self, *shape, dtype=None) -> Tensor:
        # zeros (not empty): tails that the kernels never write must stay finite
        return torch.zeros(*shape, dtype=dtype or self.dt, device=self.device)

    def _padded(self, nb: int, h: int, w: int, c: int, lo: int, hi: int) -> Tensor:
        """Interior [nb, h, w, c] view of a zero-bordered buffer (`lo` pixels before, `hi` after, rows and columns): the
        operand layout of the flat-window launches (include/bcosk.h `a_flat`).  Producers write the view, never the border."""
        buf = torch.zeros(nb, h + lo + hi, w + lo + hi, c, dtype=self.dt, device=self.device)
        return buf[:, lo:lo + h, lo:lo + w, :]

    def _dev(self, t: Tensor, dtype=torch.float32) -> Tensor:
        return t.to(device=self.device, dtype=dtype).contiguous()

    def _bn_alpha(self, prefix: str) -> Tuple[Tensor, Optional[Tensor]]:
        """eval-mode batch_norm_uncentered_2d: y = x / sqrt(running_var + eps) * weight (+ bias)."""
        var = self.sd[prefix + ".running_var"]
        w = self.sd.get(prefix + ".weight")
        alpha = 1.0 / torch.sqrt(var + self.bn_eps)
        if w is not None:
            alpha = alpha * w
        beta = self.sd.get(prefix + ".bias")
        return self._dev(alpha), (None if beta is None else self._dev(beta))

    # launches whose K loop has at most this many 64-deep stages are bandwidth bound: they use 64-wide tiles, which
    # the library runs with 3 CTAs per SM (more bytes in flight); 0 disables
    light_k_iters = 3
    parity_dgrad = True              # strided k x k data gradients as stride^2 parity-class launches (no zero insertion)
    # do not store gains that are sqrt(y / ||patch||) of a stored ReLU output.  Measured: the forward launches save 0.20 ms
    # of gain writes per step and the consumers pay 0.21 ms for the square roots (MUFU, 16 per cycle per SM): off.
    recompute_gain = False
    flat_3x3 = True                  # 64 -> <=64 channel stride-1 k x k convs and their data gradients as flat-window launches
    flat_stem = True                 # stem and its data gradient as flat-window launches (throughput mode only)
    autotune_default = True          # capture() measures the per-launch schedule first (see autotune)
    hp_wide_stages = 18  # parity-mode forward launches with at least this many (paired) K stages run 128-wide tiles (0 = never; measured: shorter
                         # K loops lose more to the exposed epilogue of the one-CTA-per-SM kernel than they gain from the smaller operand fill)
    hp_chunk = 0     # parity-mode launches: K stages per TMEM accumulation of the leading segment (0 = library default)
    fold_bn = True   # fold sqrt(BN multiplier) into the conv weights when every multiplier is positive and there is no bias

    def _block_n(self, n: int, k_iters: int = 1 << 30, hp: Optional[bool] = None) -> int:
        hp = self.hp_accum if hp is None else hp
        if n <= 32:
            return 32
        if n <= 64 or hp or k_iters <= self.light_k_iters:
            return 64
        return 128

    @staticmethod
    def _flat_fits(width: int, k: int, ntaps: int, bn: int, dense: bool, kch: int = 64) -> bool:
        """Does a flat-window launch (include/bcosk.h `a_flat`) over rows of `width` pixels (dense: the tensor's width; padded: the
        bordered buffer's pitch) fit the shared memory / TMA boxes of bcosk_igemm_flat?  Mirrors launch_flat_bn (csrc/bcosk_igemm.cu):
        wide feature maps (448^2 inputs) fall back to the im2col launches."""
        up = lambda v, a: (v + a - 1) // a * a        # noqa: E731
        row_bytes = kch * 2
        if dense:
            pitch = up(width + k - 1, 8)
            nrows = ((0 if 128 % pitch == 0 else pitch - 1) + 127) // pitch + k
            if nrows > 256 or pitch > 256:
                return False
            win = up(nrows * pitch * row_bytes, 1024)
        else:
            need = 128 + (k - 1) * width + (k - 1)
            nbox = 1 if need <= 256 else 2
            box_rows = up((need + nbox - 1) // nbox, 8)
            if box_rows > 256:
                return False
            win = up(nbox * box_rows * row_bytes, 1024)
        smem = up(ntaps * bn * row_bytes, 1024) + 2 * win + 4 * 128 * bn * 2 + 128 + 2 * bn * 4 + 2 * (bn // 32) * 128 * 4 + 64 * 4
        return smem <= 227 * 1024

    @staticmethod
    def _even_taps(wt: Tensor, taps: List[Tuple[int, int]], kch: int) -> Tuple[Tensor, List[Tuple[int, int]]]:
        """A pipeline stage is 64 K elements: with 32-channel chunks every segment needs an even number of (tap, chunk) pairs.
        An odd count (3x3 over <= 32 channels) gets one more tap that re-reads the last tap's pixels against zero weights."""
        cpt = (wt.shape[2] + kch - 1) // kch
        if kch == 32 and (len(taps) * cpt) % 2 == 1:
            wt = torch.cat([wt, wt.new_zeros(wt.shape[0], 1, wt.shape[2])], 1)
            taps = list(taps) + [taps[-1]]
        return wt, taps

    def _pack_b(self, wt: Tensor, planes: int, kch: int) -> Tuple[Tensor, int]:
        """[n, taps, c] fp32 -> (packed K-major device operand, chunks per tap).  The training plan overrides this to keep the
        operand refreshable from its fp32 master weights."""
        bmat, cpt = P.pack_b(wt, planes, kch, self.dt)
        return self._dev(bmat, self.dt), cpt

    # ------------------------------------------------------------------ forward emission
    def _conv_fwd(self, name: str, x: Act, w: Tensor, stride: int, pad_lo: int, pad_hi: int, *, bn: Optional[str],
                  relu: bool, res: Optional[Act] = None, want_mask: bool = False, y_f32: bool = False,
                  inv_norm: Optional[Tensor] = None, kch: int = 64, want_sq: bool = True,
                  sq_geom: Optional[Tuple[int, int, int, int, int]] = None, lin_bias: Optional[Tensor] = None,
                  sq_eps: Tuple[float, float] = (1e-6, 0.0), flat: bool = False, want_inv: bool = False,
                  max_out: int = 1, scale_mode: Optional[int] = None, want_gain: bool = True,
                  y_buf: Optional[Tensor] = None, y_col: int = 0, a_planes: Optional[int] = None, w_planes: Optional[int] = None,
                  y_planes: Optional[int] = None, res_planes: Optional[int] = None, hp: Optional[bool] = None,
                  out_map: Optional[Tuple[int, int, int, int]] = None, act: int = 0) -> Tuple[Act, ConvRec]:
        """One fused launch: B-cos conv (+BN multiplier, +residual, +ReLU).  The patch norm comes from `x.sq`
        (per-pixel sums of squares written by x's producer) and is evaluated inside the kernel; `sq_geom`
        overrides its (h, w, k, stride, pad) when the GEMM geometry is not the convolution's (space-to-depth stem).
        `max_out` = G > 1: the o GEMM columns are o/G groups of G adjacent units; the epilogue keeps the largest unit of each
        group, scales it and writes o/G columns (y, gain) plus the kept index (`rec.amax`), bcosconv2d.py:166-170.
        `a_planes` / `w_planes` / `y_planes` / `res_planes` (default: the plan's `planes`) give the precision planes of the input, the
        weights, the output and the residual of THIS launch (mixed formats: e.g. a one-plane branch added to a two-plane residual
        stream); `hp` overrides the choice of the fp32-faithful (plane-aware) kernel."""
        nb = self.nb
        h, wd = x.hw
        o, c, kh, kw = w.shape
        smode = self.scale_mode if scale_mode is None else scale_mode      # per-launch override (plain linear maps: NONE)
        oh = (h + pad_lo + pad_hi - kh) // stride + 1
        ow = (wd + pad_lo + pad_hi - kw) // stride + 1
        M = nb * oh * ow
        pa = self.planes if a_planes is None else a_planes
        pw = (self.fwd_w_planes or self.planes) if w_planes is None else w_planes
        segs = P.segments(pa, pw)
        hp_launch = (self.hp_accum if hp is None else hp)
        cin_phys = x.t.shape[-1] // pa
        assert c <= cin_phys
        # stride-1 k x k convs over 64 channels with <= 64 outputs (ResNet layer1 conv2): flat-window gather, the zero
        # borders are produced in shared memory by the TMA box (include/bcosk.h a_flat = 2)
        if max_out > 1:
            assert max_out in (2, 4, 8) and o % max_out == 0 and bn is None and not relu and res is None and not want_mask and not flat
        flat = flat or (self.flat_3x3 and max_out == 1 and self.planes == 1 and pa == 1 and pw == 1 and not hp_launch and stride == 1 and kh == kw and kh > 1
                        and cin_phys == 64 and kch == 64 and o <= 64 and res is None and not y_f32 and x.t.is_contiguous()
                        and self._flat_fits(wd, kh, kh * kw, 32 if o <= 32 else 64, True))
        sq_in = None
        if inv_norm is None and smode != L.BCOSK_SCALE_NONE:
            sq_in = x.sq
            if sq_geom is None:
                assert pad_lo == pad_hi and kh == kw, "asymmetric convs must pass inv_norm or sq_geom"
                sq_geom = (h, wd, kh, stride, pad_lo)
            if sq_geom[2] > 3 or flat:
                # large windows (7x7 stem: 49 taps per output pixel) are cheaper as a stand-alone sum-pool launch than as
                # 49 dependent loads in front of every tile's epilogue (measured: 9 us of a 12 us CTA lifetime)
                inv_norm = self._empty(M, dtype=torch.float32)
                self.fwd_ops.append(O.PatchNormOp(name + ".norm", x.sq, x.parts, nb, sq_geom[0], sq_geom[1], sq_geom[2],
                                                  sq_geom[3], sq_geom[4], sq_eps[0], sq_eps[1], inv_norm, oh, ow))
                sq_in = None
        alpha, beta = self._bn_alpha(bn) if bn else (None, None)
        if (alpha is not None and beta is None and self.fold_bn and smode == L.BCOSK_SCALE_B2
                and bool((alpha > 0).all())):
            # y = a * lin * |lin| / n == lin' * |lin'| / n with lin' = sqrt(a) * lin: fold sqrt(a) into the weights.  The
            # explanation pass uses the same folded weights (d y / d x = (|lin'| / n) * W'), so nothing per channel is
            # left for the epilogues.
            w = w * alpha.sqrt().to(w.device).view(-1, 1, 1, 1)
            alpha = None
        wt, taps = self._even_taps(P.fwd_weight_taps(w), P.conv_taps(kh, kw), kch)
        if (pa, pw) == (self.planes, self.planes):
            bmat, cpt = self._pack_b(wt, self.planes, kch)
        else:
            bm, cpt = P.pack_b(wt, pw, kch, self.dt, segs)
            bmat = self._dev(bm, self.dt)
        block_n = self._block_n(o, bmat.shape[1] // 64, hp=hp_launch)
        yp = 1 if y_f32 else (self.planes if y_planes is None else y_planes)
        # long K loops of the plane-aware kernel are bound by the L2 -> shared-memory operand fill (DESIGN.md 3.6): 128-wide tiles fetch the
        # A boxes once per 128 output columns (98 instead of 65 FLOP per fill byte).  Needs the packed two-plane epilogue.
        k_stages = len(taps) * cpt * kch // 64
        if (hp_launch and self.hp_wide_stages and k_stages >= self.hp_wide_stages and o % 128 == 0 and kch == 64 and yp == 2 and not y_f32
                and max_out == 1 and lin_bias is None and smode in (L.BCOSK_SCALE_B2, L.BCOSK_SCALE_NONE) and y_buf is None and out_map is None
                and (res is None or (self.planes if res_planes is None else res_planes) == 2) and segs in (P.segments(2, 2), P.segments(1, 2))
                and (not self.with_explain or not want_gain or self.gain_dt != torch.float32)):
            block_n = 128
        parts = (o + block_n - 1) // block_n
        oy = o // max_out                 # columns that leave the epilogue
        if y_buf is not None:             # the launch writes columns [y_col, y_col + oy) of every plane of a wider tensor (DenseNet features)
            assert (out_map is not None or tuple(y_buf.shape[:3]) == (nb, oh, ow)) and not y_f32 and y_buf.shape[-1] % yp == 0 and y_col % 8 == 0
            assert y_col + oy <= y_buf.shape[-1] // yp and not flat
            y = y_buf
        else:
            y = self._empty(nb, oh, ow, yp * oy, dtype=torch.float32 if y_f32 else self.dt)
        rec = ConvRec(name, w, stride, pad_lo, pad_hi, (h, wd), (oh, ow), cin_phys)
        # y = lin |lin| / n, clamped at 0: the explanation gain |lin| / n is sqrt(y / n) - not stored where that holds
        # (ReLU, no residual, BN multiplier folded, b = 2, throughput mode)
        lazy_gain = (self.with_explain and self.recompute_gain and max_out == 1 and self.planes == 1 and not self.hp_accum and relu
                     and res is None and alpha is None and beta is None and lin_bias is None and not y_f32
                     and smode == L.BCOSK_SCALE_B2)
        inv_out = None
        if lazy_gain:
            rec.gain_y = y.view(M, o)
            if inv_norm is None:
                inv_out = self._empty(M, dtype=torch.float32)
                rec.gain_inv = inv_out
            else:
                rec.gain_inv = inv_norm
        if want_inv and not lazy_gain:        # training: 1/||patch|| is needed again by the backward of the scale
            if inv_norm is None and smode != L.BCOSK_SCALE_NONE:
                inv_out = self._empty(M, dtype=torch.float32)
            rec.inv = inv_norm if inv_norm is not None else inv_out
        if self.with_explain:
            if not lazy_gain and want_gain:
                rec.gain = self._empty(M, oy, dtype=self.gain_dt)
            if max_out > 1:
                rec.amax = torch.zeros(M, oy, dtype=torch.uint8, device=self.device)
            if want_mask:
                rec.mask = self._zeros(M, (o + 31) // 32, dtype=torch.int32)
        sq = self._empty(parts, M, dtype=torch.float32) if want_sq else None
        self.fwd_ops.append(O.IgemmOp(
            name=name, a=x.t, b=bmat, n=o, lo=(-pad_lo, -pad_lo),
            up=(pad_hi - (kw - 1), pad_hi - (kh - 1)), stride=(stride, stride), op=oh, oq=ow, kch=kch, chunks_per_tap=cpt,
            taps=taps, seg_a_choff=[a * cin_phys for a, _ in segs], seg_b_plane=[b for _, b in segs], dtype=self.dt_code,
            mode=L.BCOSK_MODE_FWD, block_n=block_n, scale_mode=smode, b_exp=self.b, relu=relu,
            inv_norm=inv_norm, sq_in=sq_in, sq_geom=sq_geom, sq_eps=sq_eps, alpha=alpha, beta=beta,
            lin_bias=None if lin_bias is None else self._dev(lin_bias),
            res=None if res is None else res.t, res_planes=self.planes if res_planes is None else res_planes,
            gain=rec.gain, maskbits=rec.mask, sq_out=sq, y=y, y_planes=yp, y_f32=y_f32, hp_accum=hp_launch, hp_chunk=self.hp_chunk, flat=flat,
            inv_norm_out=inv_out, max_out=max_out, amax=rec.amax, y_col=y_col, out_map=out_map, act=act,
            algo_flops=2.0 * M * o * float((w != 0).sum().item()) / o))
        rec.algo_flops = self.fwd_ops[-1].algo_flops
        return Act(y, oy, sq, parts), rec

    # ------------------------------------------------------------------ stem of the contract-mode plans with uint8 input
    fwd_w_planes = None    # experiment knob: precision planes of the forward weights (None = the plan's planes); see scripts/exp_w_planes.py
    stem_im2col = True     # parity-mode plans with uint8 input: stem as a GEMM over an exact byte patch matrix (see _stem_fwd_im2col)

    def _stem_fwd_im2col(self, name: str, x_u8: Tensor, w: Tensor, w_s2d: Tensor, k: int, stride: int, pad: int, *, bn: Optional[str],
                         mean6, inv_std6, s2d_pad: Tuple[int, int], stem_cp: int, want_sq: bool = False) -> Tuple[Act, ConvRec]:
        """The k x k / stride stem conv + BN + ReLU of a plan whose input is uint8 RGB, in the contract (precision-plane) modes.

        The conv over the normalised [x, 1-x] input is linear in the raw bytes, so it runs as ONE 1x1 launch over the patch matrix
        `bcosk_stem_im2col_u8` writes (rows of (v_R, v_G, v_B, 1) per tap): the bytes are exact in one 16-bit plane, only the
        (folded) weights carry precision planes - `planes` plane products instead of 3 / 6, K = 256 per product instead of 512 - and
        the window is gathered once (the implicit-GEMM stem re-read its input 16 taps x 3 segments from L2: 1.95 of the 22.2 ms of
        a ResNet-50 step).  The ConvRec describes the SAME convolution in its space-to-depth form (`w_s2d`), which is what the
        explanation pass differentiates (its data gradient is unchanged)."""
        nb = self.nb
        _, _, S, _ = x_u8.shape
        o = w.shape[0]
        oh = (S + 2 * pad - k) // stride + 1
        M = nb * oh * oh
        kp = (4 * k * k + 63) // 64 * 64
        a_scale = 2.0 ** -6                       # bytes 0..255 -> 0..3.98 (exact): keeps the folded weights at the magnitude of W
        A = self._empty(nb, oh, oh, kp)
        inv = self._empty(M, dtype=torch.float32)
        self.fwd_ops.append(O.StemIm2colOp(name + ".im2col", x_u8, k, stride, pad, tuple(mean6), tuple(inv_std6), a_scale, A, inv, self.dt_code))
        alpha, beta = self._bn_alpha(bn) if bn else (None, None)
        if (alpha is not None and beta is None and self.fold_bn and self.scale_mode == L.BCOSK_SCALE_B2 and bool((alpha > 0).all())):
            sa = alpha.sqrt().to(w.device).view(-1, 1, 1, 1)          # same folding as _conv_fwd: lin' = sqrt(a) lin
            w, w_s2d = w * sa, w_s2d * sa
            alpha = None
        wf = P.stem_im2col_weight(w, mean6, inv_std6, a_scale, kp)                       # [o, kp] fp32
        planes_b = P.split_planes(wf, self.planes, self.dt)
        bmat = self._dev(torch.cat(planes_b, dim=1), self.dt)                             # [o, planes * kp]: segment s = (a plane 0, b plane s)
        y = self._empty(nb, oh, oh, self.planes * o)
        rec = ConvRec(name, w_s2d, 1, s2d_pad[0], s2d_pad[1], (oh, oh), (oh, oh), stem_cp)
        if self.with_explain:
            rec.gain = self._empty(M, o, dtype=self.gain_dt)
        block_n = self._block_n(o, self.planes * kp // 64)
        parts = (o + block_n - 1) // block_n
        sq = self._empty(parts, M, dtype=torch.float32) if want_sq else None
        self.fwd_ops.append(O.IgemmOp(
            name=name, a=A, b=bmat, n=o, lo=(0, 0), up=(0, 0), stride=(1, 1), op=oh, oq=oh, kch=64, chunks_per_tap=kp // 64, taps=[(0, 0)],
            seg_a_choff=[0] * self.planes, seg_b_plane=list(range(self.planes)), dtype=self.dt_code, mode=L.BCOSK_MODE_FWD, block_n=block_n,
            scale_mode=self.scale_mode, b_exp=self.b, relu=True, inv_norm=inv, alpha=alpha, beta=beta, gain=rec.gain, sq_out=sq, y=y,
            y_planes=self.planes, hp_accum=self.hp_accum, hp_chunk=self.hp_chunk,
            algo_flops=2.0 * M * float((w != 0).sum().item())))
        rec.algo_flops = self.fwd_ops[-1].algo_flops
        return Act(y, o, sq, parts), rec

    # ------------------------------------------------------------------ explanation emission
    @staticmethod
    def _gain_of(rec: ConvRec):
        """(mul1, mul1_sqrt_scale) the consumer's explain epilogue multiplies by: the stored gain, or the ReLU output + 1/norm"""
        return (rec.gain, None) if rec.gain is not None else (rec.gain_y, rec.gain_inv)

    def _alloc_ghat(self, rec: ConvRec, classes: bool = False) -> None:
        """Buffer for g_out * gain of `rec`.  A strided k>1 conv reads it zero-inserted at input resolution so
        that its data gradient is a stride-1 gather."""
        nb, pl = self.nb, self.bplanes
        if rec.stride > 1 and rec.k > 1 and not (classes and self.parity_dgrad):
            h, w = rec.in_hw
            assert rec.stride * (rec.out_hw[0] - 1) <= h - 1 and rec.stride * (rec.out_hw[1] - 1) <= w - 1
            rec.ghat = self._zeros(nb, h, w, pl * rec.cout)
            rec.ghat_map = (0, h * w, rec.stride * w, rec.stride)
        else:
            rec.ghat = self._zeros(nb, rec.out_hw[0], rec.out_hw[1], pl * rec.cout)
            rec.ghat_map = None

    def _dgrad(self, rec: ConvRec, *, y: Tensor, y_map=None, mul1: Optional[Tensor] = None, add: Optional[Tensor] = None,
               add_stride: int = 1, out2: Optional[Tensor] = None, mul2: Optional[Tensor] = None,
               mask2: Optional[Tensor] = None, y_f32: bool = False, kch: int = 64, flat: bool = False,
               mul1_sqrt_scale: Optional[Tensor] = None) -> None:
        """Data gradient of `rec` as a stride-1 gather over rec.ghat (tcgen05 implicit GEMM, explain epilogue)."""
        g = rec.ghat
        k = rec.k
        if rec.stride > 1 and k > 1 and rec.ghat_map is None:
            assert add is None and out2 is None and y_map is None and not y_f32 and not flat
            return self._dgrad_classes(rec, y=y, mul1=mul1, kch=kch, mul1_sqrt_scale=mul1_sqrt_scale)
        if rec.stride > 1 and k == 1:
            oh, ow = rec.out_hw      # dense GEMM at output resolution; consumer adds it sub-sampled
        else:
            oh, ow = rec.in_hw
        flat = flat or (self.flat_3x3 and self.bplanes == 1 and not self.bwd_hp and rec.stride == 1 and k > 1
                        and rec.cout == 64 and kch == 64 and rec.cin_phys <= 64 and add is None and out2 is None
                        and y_map is None and not y_f32 and g.is_contiguous()
                        and self._flat_fits(g.shape[2], k, k * k, 32 if rec.cin_phys <= 32 else 64, True))
        lo = rec.pad_lo - (k - 1)
        up_h = oh - g.shape[1] + lo
        up_w = ow - g.shape[2] + lo
        n = rec.cin_phys
        wt = P.dgrad_weight_taps(rec.w)                      # [c, taps, o]
        if wt.shape[0] < n:                                  # physical input channels beyond the logical ones
            wt = torch.cat([wt, wt.new_zeros(n - wt.shape[0], *wt.shape[1:])], 0)
        wt, taps = self._even_taps(wt, P.conv_taps(k, k), kch)
        bmat, cpt = self._pack_b(wt, self.bplanes, kch)
        self.bwd_ops.append(O.IgemmOp(
            name=rec.name + ".dgrad", a=g, b=bmat, n=n, lo=(lo, lo), up=(up_w, up_h), stride=(1, 1),
            op=oh, oq=ow, kch=kch, chunks_per_tap=cpt, taps=taps,
            seg_a_choff=P.seg_a_offsets(self.bplanes, rec.cout), seg_b_plane=P.seg_b_planes(self.bplanes), dtype=self.dt_code, mode=L.BCOSK_MODE_EXPLAIN,
            block_n=64 if (add is not None and add_stride == 1 and self.bplanes == 1 and n >= 64)
            else self._block_n(n, bmat.shape[1] // 64, hp=self.bwd_hp),   # dense extra gradient: 64-wide tiles stage it with TMA
            hp_accum=self.bwd_hp, hp_chunk=self.hp_chunk, y=y, y_planes=1 if y_f32 else self.bplanes, y_f32=y_f32,
            out_map=y_map, add=add, add_planes=self.bplanes, add_stride=add_stride, mul1=mul1, out2=out2,
            out2_planes=self.bplanes, mul2=mul2, mask2=mask2, flat=flat, mul1_sqrt_scale=mul1_sqrt_scale,
            algo_flops=rec.algo_flops,
            a_dense_frac=1.0 / (rec.stride * rec.stride) if rec.ghat_map is not None else 1.0))

    def _dgrad_classes(self, rec: ConvRec, *, y: Tensor, mul1: Optional[Tensor], kch: int = 64,
                       mul1_sqrt_scale: Optional[Tensor] = None) -> None:
        """Strided k x k data gradient over the DENSE gradient tensor, one launch per parity class of the input pixel.

        gx[s*i+py, s*j+px] = sum over the taps dy = ry + s*t (ry = (py+pad) % s) of g[i + cy - t, ...] W[dy, dx]^T with
        cy = (py + pad - ry) / s: a stride-1 gather with Ty x Tx taps whose lower corner is cy - (Ty - 1).  The s*s launches
        do k*k/(s*s) taps per input pixel; a zero-inserted gradient would cost k*k (include/bcosk.h `side_mapped`)."""
        g = rec.ghat
        k, s, pad = rec.k, rec.stride, rec.pad_lo
        assert rec.pad_lo == rec.pad_hi
        ih, iw = rec.in_hw
        n = rec.cin_phys
        nz = float((rec.w != 0).sum().item())
        for py in range(s):
            ry = (py + pad) % s
            dys = list(range(ry, k, s))
            cy = (py + pad - ry) // s
            for px in range(s):
                rx = (px + pad) % s
                dxs = list(range(rx, k, s))
                cx = (px + pad - rx) // s
                ty, tx = len(dys), len(dxs)
                assert ty > 0 and tx > 0, "a parity class without taps (k < stride) is not handled here"
                oh, ow = (ih - py + s - 1) // s, (iw - px + s - 1) // s
                lo_h, lo_w = cy - (ty - 1), cx - (tx - 1)
                # tap (jx, jy) reads g[i + lo_h + jy] -> t = ty - 1 - jy -> dy = ry + s * (ty - 1 - jy)
                sel = [(dys[ty - 1 - jy], dxs[tx - 1 - jx]) for jy in range(ty) for jx in range(tx)]
                wt = torch.stack([rec.w[:, :, dy, dx].t() for dy, dx in sel], 1)       # [c, taps, o]
                if wt.shape[0] < n:
                    wt = torch.cat([wt, wt.new_zeros(n - wt.shape[0], *wt.shape[1:])], 0)
                bmat, cpt = self._pack_b(wt, self.bplanes, kch)
                self.bwd_ops.append(O.IgemmOp(
                    name=f"{rec.name}.dgrad.c{py}{px}", a=g, b=bmat, n=n, lo=(lo_w, lo_h),
                    up=(ow - g.shape[2] + lo_w, oh - g.shape[1] + lo_h), stride=(1, 1), op=oh, oq=ow, kch=kch,
                    chunks_per_tap=cpt, taps=[(jx, jy) for jy in range(ty) for jx in range(tx)],
                    seg_a_choff=P.seg_a_offsets(self.bplanes, rec.cout), seg_b_plane=P.seg_b_planes(self.bplanes), dtype=self.dt_code, mode=L.BCOSK_MODE_EXPLAIN,
                    block_n=self._block_n(n, bmat.shape[1] // 64, hp=self.bwd_hp), hp_accum=self.bwd_hp, hp_chunk=self.hp_chunk, y=y, y_planes=self.bplanes,
                    out_map=(py * iw + px, ih * iw, s * iw, s), mul1=mul1, side_mapped=True, mul1_sqrt_scale=mul1_sqrt_scale,
                    algo_flops=rec.algo_flops * (sum(float((rec.w[:, :, dy, dx] != 0).sum().item()) for dy, dx in sel) / nz),
                    a_dense_frac=1.0 / (s * s)))    # the s*s launches together read the gradient once

    # ------------------------------------------------------------------ execution
    def _require_gpu(self) -> None:
        if self.device.type != "cuda":
            raise L.BcoskError("plans execute only on a CUDA device (sm_100a); no CPU fallback exists")
        L.require_device()

    def run_forward(self) -> None:
        self._require_gpu()
        O.run_ops(self.fwd_ops)

    def run_explain(self) -> None:
        self._require_gpu()
        O.run_ops(self.bwd_ops)

    def autotune(self, reps: int = 5) -> dict:
        """Pick the schedule (include/bcosk.h `sched`) of every 64-wide tensor-core launch, and the tile width (64 / 128) of
        the launches that write no per-tile sums of squares, by measuring each candidate in place.

        The three schedules give bit-identical outputs (tests/test_kernels_gpu.py); which is fastest depends on N, K and
        the epilogue streams (measured: profiles/r01_schedule_ab.md), so it is decided per launch, once, before capture.
        64-wide forward launches of the plane-aware kernel (hp_accum) choose between two (sched 1), three (sched 3) and four
        (sched 4) CTAs per SM, which also give bit-identical outputs (tests/test_igemm_hp_ctas_gpu.py; profiles/r03_hp_three_ctas.md).
        Returns {launch name: (block_n, sched)}.
        """
        self._require_gpu()
        self.run_forward()
        if self.with_explain:
            self.run_explain()
        torch.cuda.synchronize()
        chosen = {}
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]

        def timed(op) -> float:
            op.run()
            ts = []
            for _ in range(reps):
                ev[0].record()
                op.run()
                ev[1].record()
                ev[1].synchronize()
                ts.append(ev[0].elapsed_time(ev[1]))
            return sorted(ts)[len(ts) // 2]

        for op in self.fwd_ops + (self.bwd_ops if self.with_explain else []):
            if not isinstance(op, O.IgemmOp) or op.flat:
                continue
            if op.hp_accum:
                # plane-aware kernel: 64-wide forward launches run two (sched 1), three (sched 3) or four (sched 4) CTAs per SM
                if op.mode != L.BCOSK_MODE_FWD or op.resolved_block_n() != 64:
                    continue
                cands = [(64, 1), (64, 3), (64, 4)]
            else:
                # tile width: free to choose where no per-tile partial sums of squares are written (their layout follows it)
                widths = [op.resolved_block_n()]
                if op.sq_out is None and op.n >= 128 and widths[0] in (64, 128):
                    widths = [64, 128]
                if widths == [128]:
                    continue
                cands = [(bn, sched) for bn in widths for sched in ((1, 2, 3) if bn == 64 else (0,))
                         if not (sched == 3 and op.n <= 64)]   # a single n tile: 3 is the same as 2
            best, best_t = cands[0], float("inf")
            for bn, sched in cands:
                op.block_n, op.sched = bn, sched
                t = timed(op)
                if t < best_t * 0.98:                 # prefer the earlier (simpler) candidate on a tie
                    best, best_t = (bn, sched), t
            op.block_n, op.sched = best
            chosen[op.name] = best
            op.run()                                  # leave the tensors as the chosen configuration writes them
        self.schedules = chosen
        return chosen

    def capture(self, autotune: Optional[bool] = None) -> None:
        """Capture forward and forward+explain as CUDA graphs (kernel parameters incl. TMA descriptors are baked in)."""
        self._require_gpu()
        if self.autotune_default if autotune is None else autotune:
            self.autotune()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            self.run_forward()
            if self.with_explain:
                self.run_explain()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        self._graph_fwd = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._graph_fwd):
            O.run_ops(self.fwd_ops)
        if self.with_explain:
            self._graph_all = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self._graph_all):
                O.run_ops(self.fwd_ops)
                O.run_ops(self.bwd_ops)
            self._graph_bwd = torch.cuda.CUDAGraph()      # explanation pass alone: further targets reuse one forward
            with torch.cuda.graph(self._graph_bwd):
                O.run_ops(self.bwd_ops)

    def replay_forward(self) -> None:
        if self._graph_fwd is not None:
            self._graph_fwd.replay()
        else:
            self.run_forward()

    def replay_explain(self) -> None:
        if self._graph_bwd is not None:
            self._graph_bwd.replay()
        else:
            self.run_explain()

    def replay_all(self) -> None:
        if self._graph_all is not None:
            self._graph_all.replay()
        else:
            self.run_forward()
            self.run_explain()

    # ------------------------------------------------------------------ accounting
    def num_launches(self, explain: bool = True) -> int:
        return len(self.fwd_ops) + (len(self.bwd_ops) if explain else 0)

    def gemm_flops(self, explain: bool = True) -> float:
        ops = self.fwd_ops + (self.bwd_ops if explain else [])
        return sum(o.flops() for o in ops if isinstance(o, O.IgemmOp))
