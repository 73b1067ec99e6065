"""Launch records of the fused execution plans.

A plan is a flat list of these records; each one names the device tensors it reads/writes and maps
1:1 onto one entry point of the C ABI (include/bcosk.h).  `run()` enqueues the kernel on the current
CUDA stream through ctypes - there is no other execution path in the product (tests/emulator.py holds
a torch restatement of each record's semantics that is used ONLY to check plans on CPU).
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import List, Optional, Tuple

import torch
from torch import Tensor

from .. import _lib as L


@dataclass
class IgemmOp:
    """One `bcosk_igemm` launch (forward B-cos epilogue or explain-dgrad epilogue)."""
    name: str
    a: Tensor                      # [nb, h, w, a_c] 16-bit NHWC (a_c = planes * channels)
    b: Tensor                      # [n, ktot] packed weights
    n: int
    lo: Tuple[int, int]            # (w, h) lower corner
    up: Tuple[int, int]
    stride: Tuple[int, int]
    op: int
    oq: int
    kch: int
    chunks_per_tap: int
    taps: List[Tuple[int, int]]    # (off_w, off_h)
    seg_a_choff: List[int]
    dtype: int
    seg_b_plane: Optional[List[int]] = None   # B plane per segment (engine/pack.py SEGMENTS); None = [0] for one segment
    mode: int = 0
    block_n: int = 0
    # forward epilogue
    scale_mode: int = 0
    b_exp: float = 2.0
    relu: bool = False
    inv_norm: Optional[Tensor] = None      # [M] precomputed 1/||patch||, or None -> computed in-kernel from sq_in
    sq_in: Optional[Tensor] = None         # [parts, nb*sq_h*sq_w] per-pixel sums of squares of the input tensor
    sq_geom: Optional[Tuple[int, int, int, int, int]] = None   # (sq_h, sq_w, k, stride, pad)
    sq_eps: Tuple[float, float] = (1e-6, 0.0)                   # (inside sqrt, outside sqrt)
    alpha: Optional[Tensor] = None
    beta: Optional[Tensor] = None
    lin_bias: Optional[Tensor] = None      # [n] fp32 bias of the linear map (added before the scale)
    res: Optional[Tensor] = None
    res_planes: int = 1
    gain: Optional[Tensor] = None
    maskbits: Optional[Tensor] = None
    sq_out: Optional[Tensor] = None
    # primary output
    y: Optional[Tensor] = None
    y_planes: int = 1
    y_f32: bool = False
    out_map: Optional[Tuple[int, int, int, int]] = None   # (os_0, os_n, os_p, os_q); None = dense
    # explain epilogue
    add: Optional[Tensor] = None
    add_planes: int = 1
    add_stride: int = 1
    mul1: Optional[Tensor] = None
    out2: Optional[Tensor] = None
    out2_planes: int = 1
    mul2: Optional[Tensor] = None
    mask2: Optional[Tensor] = None
    # accounting (set by the plan): 2*MAC of the logical convolution, fraction of `a` that is not structural zeros
    algo_flops: float = 0.0
    a_dense_frac: float = 1.0
    hp_accum: bool = False           # per-stage TMEM accumulators summed in registers (parity mode)
    hp_chunk: int = 0                # include/bcosk.h `hp_chunk`: K stages per TMEM accumulation of the leading segment (0 = default)
    sched: int = 0                   # include/bcosk.h `sched`: 0 / 1 per tile, 2 persistent, 3 persistent row blocks
                                     # (hp_accum forward launches: 3 / 4 = three / four CTAs per SM, else two)
    flat: bool = False               # include/bcosk.h `a_flat`: `a` is the interior view of a zero-bordered buffer
    side_mapped: bool = False        # include/bcosk.h `side_mapped`: mul1 / out2 / ... follow the mapped output row
    inv_norm_out: Optional[Tensor] = None      # forward: [M] fp32, receives the 1/||patch|| the launch used
    mul1_sqrt_scale: Optional[Tensor] = None   # explain: mul1 holds the producer's ReLU output, gain = sqrt(mul1 * this[row])
    y_col: int = 0                             # first column of the n-column slice of `y` this launch writes in every plane (DenseNet
                                               # feature tensors: y = the whole block tensor, y_ld = its row pitch); 0 = y is the launch's own
    max_out: int = 1                           # include/bcosk.h `max_out`: groups of adjacent units reduced in the forward epilogue
    amax: Optional[Tensor] = None              # [M, n / max_out] uint8: index of the kept unit
    act: int = 0                               # include/bcosk.h `act`: 1 = MyGELU, 2 = QuickGELU behind the transform (folded into y and the gain)

    # ---- derived ----
    @property
    def M(self) -> int:
        return self.a.shape[0] * self.op * self.oq

    @property
    def ktot(self) -> int:
        return len(self.seg_a_choff) * len(self.taps) * self.chunks_per_tap * self.kch

    def flops(self) -> float:
        return 2.0 * self.M * self.n * self.ktot

    def smem_fill_bytes(self) -> float:
        """Operand bytes the launch's TMA loads move from L2 into shared memory over its K loops, per-tile schedule: every (m tile, n tile)
        pair fetches its A boxes (once per distinct a-plane in the paired stages of the plane-aware kernel, else once per segment) and its
        B boxes (once per segment).  The L2 -> SM path (LTS cap, B300_MICROARCH.md) is what bounds the K >= 1024 contract-mode launches."""
        bn = self.resolved_block_n()
        m_tiles, n_tiles = (self.M + 127) // 128, (self.n + bn - 1) // bn
        k_seg = len(self.taps) * self.chunks_per_tap * self.kch
        segs = len(self.seg_a_choff)
        sb = list(self.seg_b_plane or [0])
        paired = (self.hp_accum and self.kch == 64 and segs >= 2 and sb[:2] == [0, 1] and self.seg_a_choff[0] == self.seg_a_choff[1]
                  and (segs == 2 or (segs == 3 and sb[2] == 0 and self.seg_a_choff[2] != self.seg_a_choff[0])))
        a_loads = len(set(self.seg_a_choff)) if paired else segs
        b_loads = 2 if paired else segs
        return float(m_tiles) * n_tiles * (a_loads * 128 + b_loads * bn) * k_seg * 2.0

    def algo_bytes(self) -> float:
        """Algorithmic HBM bytes of this launch: every operand / result tensor moved exactly once
        (x, W, y, gain, mask, sq, residual | g_out, W, g_in, gains, masks, extra gradient)."""
        def nbytes(t):
            return 0.0 if t is None else float(t.numel() * t.element_size())
        nb, h, w, ac = self.a.shape
        strided_1x1 = len(self.taps) == 1 and self.stride[0] > 1
        a_pix = self.M if strided_1x1 else nb * h * w
        total = a_pix * ac * self.a.element_size() * self.a_dense_frac
        total += nbytes(self.b)
        ywidth = self.y.shape[-1] if (self.y_col == 0 and self.max_out == 1 and self.y.shape[-1] <= (1 if self.y_f32 else self.y_planes) * self.n) \
            else (1 if self.y_f32 else self.y_planes) * (self.n // max(self.max_out, 1))
        ydense = self.M * ywidth * self.y.element_size()      # rows actually written
        total += ydense
        if self.inv_norm is None and self.sq_in is not None:
            total += nbytes(self.sq_in)
        for t in (self.inv_norm, self.alpha, self.beta, self.res, self.gain, self.maskbits, self.sq_out, self.add,
                  self.inv_norm_out, self.mul1_sqrt_scale):
            total += nbytes(t)
        for t in (self.mul1, self.out2, self.mul2, self.mask2):
            if t is not None and self.side_mapped:      # a parity-class launch touches only its own rows of these
                total += float(self.M * t.shape[-1] * t.element_size())
            else:
                total += nbytes(t)
        return total

    def flat_geometry(self) -> Tuple[int, int, int, int]:
        """(row pitch, image pitch in rows, window origin, buffer size) in pixels of the zero-bordered buffer behind `a`."""
        nb, h, w, ac = self.a.shape
        s_n, s_h, s_w, s_c = self.a.stride()
        assert s_c == 1 and s_w == ac and s_h % ac == 0 and s_n % s_h == 0, (self.name, "not a padded NHWC view")
        wp, hp = s_h // ac, s_n // s_h
        base = self.a._base if self.a._base is not None else self.a
        assert self.a.storage_offset() % ac == 0
        off = self.a.storage_offset() // ac
        top, left = off // wp, off % wp
        kw = max(t[0] for t in self.taps) + 1
        kh = max(t[1] for t in self.taps) + 1
        lo_w, lo_h = self.lo
        assert left >= -lo_w and wp - w - left >= kw - 1 + lo_w, (self.name, "horizontal border too narrow")
        assert top >= -lo_h and hp - h - top >= kh - 1 + lo_h, (self.name, "vertical border too narrow")
        assert self.stride == (1, 1) and len(self.seg_a_choff) == 1 and self.chunks_per_tap == 1 and self.n <= 64
        return wp, hp, off + lo_h * wp + lo_w, base.numel() // ac

    def resolved_block_n(self) -> int:
        if self.block_n:
            return self.block_n
        return 32 if self.n <= 32 else (64 if (self.n <= 64 or self.hp_accum) else 128)

    def params(self) -> L.IgemmParams:
        p = L.IgemmParams()
        nb, h, w, ac = self.a.shape
        p.a = self.a.data_ptr()
        p.a_nb, p.a_h, p.a_w, p.a_c = nb, h, w, ac
        p.lo_w, p.lo_h = self.lo
        p.up_w, p.up_h = self.up
        p.stride_w, p.stride_h = self.stride
        p.op, p.oq = self.op, self.oq
        p.kch, p.chunks_per_tap = self.kch, self.chunks_per_tap
        p.num_taps, p.num_segs = len(self.taps), len(self.seg_a_choff)
        for i, o in enumerate(self.seg_a_choff):
            p.seg_a_choff[i] = o
        for i, bp in enumerate(self.seg_b_plane or []):
            p.seg_b_plane[i] = bp
        for i, (ow, oh) in enumerate(self.taps):
            p.tap_off_w[i], p.tap_off_h[i] = ow, oh
        assert self.b.shape == (self.n, self.ktot), (self.name, self.b.shape, self.n, self.ktot)
        p.b = self.b.data_ptr()
        p.n, p.dtype, p.block_n, p.mode = self.n, self.dtype, self.resolved_block_n(), self.mode
        p.scale_mode, p.b_exp, p.relu = self.scale_mode, self.b_exp, int(self.relu)
        p.set_ptr("inv_norm", self.inv_norm)
        if self.inv_norm is None and self.sq_in is not None:
            p.sq_in = self.sq_in.data_ptr()
            p.sq_parts = self.sq_in.shape[0]
            p.sq_h, p.sq_w, p.sq_k, p.sq_stride, p.sq_pad = self.sq_geom
            p.sq_eps_in, p.sq_eps_out = self.sq_eps
        p.set_ptr("alpha", self.alpha)
        p.set_ptr("beta", self.beta)
        p.set_ptr("lin_bias", self.lin_bias)
        if self.res is not None:
            p.res = self.res.data_ptr()
            p.res_ld = self.res.shape[-1]
            p.res_planes = self.res_planes
            p.res_plane_stride = self.res.shape[-1] // self.res_planes
        if self.gain is not None:
            p.gain = self.gain.data_ptr()
            p.gain_ld = self.gain.shape[-1]
            p.gain_f32 = int(self.gain.dtype == torch.float32)
        if self.maskbits is not None:
            p.maskbits = self.maskbits.data_ptr()
            p.mask_ld = self.maskbits.shape[-1]
        p.set_ptr("sq_out", self.sq_out)
        p.y = self.y.data_ptr() + self.y_col * self.y.element_size()
        p.y_ld = self.y.shape[-1]
        p.y_planes = self.y_planes
        p.y_plane_stride = self.y.shape[-1] // self.y_planes
        p.y_f32 = int(self.y_f32)
        if self.out_map is None:
            p.os_0, p.os_n, p.os_p, p.os_q = 0, self.op * self.oq, self.oq, 1
        else:
            p.os_0, p.os_n, p.os_p, p.os_q = self.out_map
        if self.add is not None:
            p.add = self.add.data_ptr()
            p.add_ld = self.add.shape[-1]
            p.add_planes = self.add_planes
            p.add_plane_stride = self.add.shape[-1] // self.add_planes
            p.add_stride = self.add_stride
            p.add_p, p.add_q = self.add.shape[1], self.add.shape[2]
        if self.mul1 is not None:
            p.mul1 = self.mul1.data_ptr()
            p.mul1_ld = self.mul1.shape[-1]
            p.mul1_f32 = int(self.mul1.dtype == torch.float32)
        if self.out2 is not None:
            p.out2 = self.out2.data_ptr()
            p.out2_ld = self.out2.shape[-1]
            p.out2_planes = self.out2_planes
            p.out2_plane_stride = self.out2.shape[-1] // self.out2_planes
        if self.mul2 is not None:
            p.mul2 = self.mul2.data_ptr()
            p.mul2_ld = self.mul2.shape[-1]
            p.mul2_f32 = int(self.mul2.dtype == torch.float32)
        if self.mask2 is not None:
            p.mask2 = self.mask2.data_ptr()
            p.mask2_ld = self.mask2.shape[-1]
        p.hp_accum = int(self.hp_accum)
        p.hp_chunk = int(self.hp_chunk)
        p.sched = int(self.sched)
        p.side_mapped = int(self.side_mapped)
        p.set_ptr("inv_norm_out", self.inv_norm_out)
        p.set_ptr("mul1_sqrt_scale", self.mul1_sqrt_scale)
        p.act = int(self.act)
        if self.max_out > 1:
            p.max_out = self.max_out
            if self.amax is not None:
                p.amax, p.amax_ld = self.amax.data_ptr(), self.amax.shape[-1]
        if self.flat and self.a.is_contiguous():
            p.a_flat = 2                      # dense tensor: the zero borders are made in shared memory
            assert self.stride == (1, 1) and len(self.seg_a_choff) == 1 and self.chunks_per_tap == 1 and self.n <= 64
        elif self.flat:
            wp, hp, origin, total = self.flat_geometry()
            p.a_flat, p.a_wp, p.a_hp, p.a_flat_rows = 1, wp, hp, total - origin
        return p

    def run(self) -> None:
        L.igemm(self.params())


@dataclass
class InputPrepOp:
    name: str
    x: Tensor            # [nb, 6, h, w] fp32
    mean6: Tuple[float, ...]
    inv_std6: Tuple[float, ...]
    out: Tensor          # [nb, h/2, w/2, planes*cp]
    cp: int
    planes: int
    dtype: int
    sq: Optional[Tensor]  # [nb*h*w] fp32

    def run(self) -> None:
        L.input_prep_s2d(self.x, self.mean6, self.inv_std6, self.out, self.cp, self.planes, self.dtype, self.sq)


@dataclass
class PatchNormOp:
    name: str
    sq: Tensor           # [parts, nb*h*w] fp32
    parts: int
    nb: int
    h: int
    w: int
    k: int
    stride: int
    pad: int
    eps_in: float
    eps_out: float
    inv_norm: Tensor     # [nb*op*oq]
    op: int
    oq: int

    def run(self) -> None:
        L.patch_inv_norm(self.sq, self.parts, self.nb, self.h, self.w, self.k, self.k, self.stride, self.pad, self.eps_in,
                         self.eps_out, self.inv_norm, self.op, self.oq)


@dataclass
class AvgPoolFwdOp:
    name: str
    x: Tensor            # [nb, h, w, planes*c]
    c: int
    planes: int
    k: int
    stride: int
    pad: int
    y: Tensor            # [nb, op, oq, planes*c]
    dtype: int
    sq: Optional[Tensor]

    def run(self) -> None:
        nb, h, w, _ = self.x.shape
        L.avgpool_fwd(self.x, nb, h, w, self.c, self.planes, self.k, self.stride, self.pad, self.y, self.y.shape[1],
                      self.y.shape[2], self.dtype, self.sq)


@dataclass
class AvgPoolBwdMulOp:
    name: str
    gy: Tensor           # [nb, op, oq, planes*c]
    c: int
    planes: int
    k: int
    stride: int
    pad: int
    gain: Optional[Tensor]  # [nb*h*w, c]
    gx: Tensor           # [nb, h, w, planes*c]
    dtype: int
    gain_sqrt_scale: Optional[Tensor] = None   # [nb*h*w] fp32: `gain` holds the ReLU output y, multiplier = sqrt(y * this)

    def run(self) -> None:
        nb, h, w, _ = self.gx.shape
        L.avgpool_bwd_mul(self.gy, nb, h, w, self.c, self.planes, self.k, self.stride, self.pad, self.gy.shape[1],
                          self.gy.shape[2], self.gain, self.gain is not None and self.gain.dtype == torch.float32,
                          self.gx, self.dtype, self.gain_sqrt_scale)


@dataclass
class GapLogitsOp:
    name: str
    fc: Tensor           # [nb*npix, ncls] fp32
    nb: int
    npix: int
    ncls: int
    inv_temp: float
    bias: float
    logits: Tensor       # [nb, ncls] fp32
    pred: Tensor         # [nb] int32

    def run(self) -> None:
        L.gap_logits(self.fc, self.nb, self.npix, self.ncls, self.inv_temp, self.bias, self.logits, self.pred)


@dataclass
class FcSeedOp:
    name: str
    target: Tensor       # [nb] int32
    gain_fc: Tensor      # [nb*npix, ncls]
    w_fc: Tensor         # [ncls, c] fp32
    nb: int
    npix: int
    ncls: int
    c: int
    inv_temp: float
    seed_scale: float
    mul1: Optional[Tensor]
    out1: Tensor         # [nb*npix, planes*c]
    mask2: Optional[Tensor]
    out2: Optional[Tensor]
    planes: int
    dtype: int

    def run(self) -> None:
        L.fc_seed_dgrad(self.target, self.gain_fc, self.gain_fc.dtype == torch.float32, self.w_fc, self.nb, self.npix,
                        self.ncls, self.c, self.inv_temp, self.seed_scale, self.mul1,
                        self.mul1 is not None and self.mul1.dtype == torch.float32, self.out1, self.mask2, self.out2,
                        self.planes, self.dtype)


@dataclass
class ContribMapOp:
    name: str
    g: Tensor            # [nb, h/2, w/2, cp] fp32 (space-to-depth stem gradient)
    x: Tensor            # [nb, 6, h, w] fp32
    cp: int
    inv_std6: Tuple[float, ...]
    out_scale: float
    cmap: Tensor         # [nb, h, w] fp32
    grad6: Optional[Tensor]  # [nb, 6, h, w] fp32

    def run(self) -> None:
        nb, _, h, w = self.x.shape
        L.contrib_map_s2d(self.g, self.x, nb, h, w, self.cp, self.inv_std6, self.out_scale, self.cmap, self.grad6)


@dataclass
class ExplanationImageOp:
    """RGBA explanation images of the batch (gradient_to_image, bcos/common.py:387-436) from grad6 and the input."""
    name: str
    grad6: Tensor        # [nb, 6, h, w] fp32 dynamic linear weights
    x: Tensor            # [nb, 6, h, w] fp32 or uint8 RGB [nb, 3, h, w]
    smooth: int
    percentile: float
    tmp: Tensor          # [2*nb*h*w + nb] fp32 scratch
    out: Tensor          # [nb, h, w, 4] fp32

    def run(self) -> None:
        L.explanation_rgba(self.grad6, self.x, self.smooth, self.percentile, self.tmp, self.out)


@dataclass
class TrunkOutOp:
    """Trunk output NHWC 16-bit planes -> NCHW fp32 (the layout the module-level head reads)."""
    name: str
    y: Tensor
    nb: int
    c: int
    h: int
    w: int
    planes: int
    dtype: int
    out: Tensor

    def run(self) -> None:
        L.nhwc_to_nchw_f32(self.y, self.nb, self.c, self.h, self.w, self.planes, self.dtype, self.out)


@dataclass
class SeedFromNchwOp:
    """include/bcosk.h bcosk_seed_from_nchw: external gradient (NCHW fp32) -> last block's ghat (x gain) and side (masked)."""
    name: str
    g: Tensor
    seed_scale: float
    mul1: Optional[Tensor]
    out1: Tensor
    mask2: Optional[Tensor]
    mul2: Optional[Tensor]
    out2: Optional[Tensor]
    planes: int
    dtype: int

    def run(self) -> None:
        L.seed_from_nchw(self.g, self.seed_scale, self.mul1, self.out1, self.mask2, self.mul2, self.out2, self.planes, self.dtype)


# ---------------------------------------------------------------------------------------------------------------------
# Fused SimpleViT plan (engine/vit.py; kernels: csrc/bcosk_vit.cu).  Token tensors: [nb, gh, gw, planes * d].
# ---------------------------------------------------------------------------------------------------------------------
@dataclass
class VitPatchifyOp:
    name: str
    x: Tensor            # [nb, 6, h, w] fp32 or uint8 RGB [nb, 3, h, w]
    p: int
    mean6: Tuple[float, ...]
    inv_std6: Tuple[float, ...]
    out: Tensor          # [nb, h/p, w/p, planes * p*p*6]
    planes: int
    dtype: int
    sq: Optional[Tensor]  # [1, rows] fp32

    def run(self) -> None:
        L.vit_patchify(self.x, self.p, self.mean6, self.inv_std6, self.out, self.planes, self.dtype, self.sq)


@dataclass
class VitContribMapOp:
    name: str
    g: Tensor            # [nb, gh, gw, p*p*6] fp32 (patch-embedding data gradient)
    x: Tensor
    p: int
    inv_std6: Tuple[float, ...]
    out_scale: float
    cmap: Tensor         # [nb, h, w] fp32
    grad6: Optional[Tensor]

    def run(self) -> None:
        L.vit_contrib_map(self.g, self.x, self.p, self.inv_std6, self.out_scale, self.cmap, self.grad6)


@dataclass
class VitLnFwdOp:
    name: str
    x: Tensor            # [.., planes * d]
    d: int
    planes: int
    w: Tensor            # [d] fp32
    eps: float
    y: Tensor
    rstd: Tensor         # [rows] fp32
    sq: Optional[Tensor]  # [1, rows] fp32: sum of the stored outputs squared
    dtype: int
    out_planes: int = 0  # planes of y (0 = `planes`)

    def run(self) -> None:
        L.vit_ln_fwd(self.x, self.rstd.numel(), self.d, self.planes, self.w, self.eps, self.y, self.rstd, self.sq, self.dtype, self.out_planes)


@dataclass
class VitLnBwdOp:
    """G_out = G_in + rstd * (g w - mean(g w));  ghat = G_out * gain (one 16-bit plane)."""
    name: str
    g: Tensor            # [.., d] fp32 or 16-bit
    G_in: Optional[Tensor]   # [.., d] fp32
    d: int
    w: Tensor
    rstd: Tensor
    G_out: Optional[Tensor]  # fp32
    gain: Optional[Tensor]
    ghat: Optional[Tensor]   # 16-bit
    dtype: int
    x: Optional[Tensor] = None   # TRUE backward (nothing detached; CLIP's LayerNorm): the LayerNorm input as plane rows
    x_planes: int = 1

    def run(self) -> None:
        if self.x is not None:
            L.vit_ln_bwd_full(self.g, self.x, self.x_planes, self.G_in, self.rstd.numel(), self.d, self.w, self.rstd, self.G_out, self.gain,
                              self.ghat, self.dtype)
        else:
            L.vit_ln_bwd(self.g, self.G_in, self.rstd.numel(), self.d, self.w, self.rstd, self.G_out, self.gain, self.ghat, self.dtype)


@dataclass
class VitGeluFwdOp:
    name: str
    u: Tensor            # [.., planes * d]
    d: int
    planes: int
    a: Tensor
    sq: Optional[Tensor]
    gain: Optional[Tensor]   # [rows, d] multiplied in place by the gate
    dtype: int
    quick: bool = False      # CLIP's QuickGELU (u sigmoid(1.702 u)); the gain is multiplied by its TRUE derivative (not detached there)

    def run(self) -> None:
        fn = L.vit_quickgelu_fwd if self.quick else L.vit_gelu_fwd
        fn(self.u, self.u.numel() // self.u.shape[-1], self.d, self.planes, self.a, self.sq, self.gain, self.dtype)


@dataclass
class VitAttentionOp:
    name: str
    qkv: Tensor          # [nb, gh, gw, planes * 3*heads*dh]
    planes: int
    g: Optional[Tensor]  # backward: [nb, gh, gw, heads*dh] fp32
    nb: int
    n: int
    heads: int
    dh: int
    scale: float
    backward: bool
    out: Tensor          # forward: planes * heads*dh; backward: heads*dh (one plane)
    dtype: int
    tc: bool = True      # tensor-core kernel (bcosk_vit_attention_tc); False = the CUDA-core shared-memory kernel (n <= 208)
    full_bwd: bool = False   # backward with NOTHING frozen (CLIP's nn.MultiheadAttention): out = [.., 3*heads*dh] (dq | dk | dv), one plane

    def run(self) -> None:
        if self.backward and self.full_bwd:
            L.vit_attention_bwd_full(self.qkv, self.planes, self.g, self.nb, self.n, self.heads, self.dh, self.scale, self.out, self.dtype)
            return
        L.vit_attention(self.qkv, self.planes, self.g, self.nb, self.n, self.heads, self.dh, self.scale, self.backward, self.out, self.dtype,
                        self.tc)


@dataclass
class PixelSqsumOp:
    """sq[row] = sum over the columns of a plane row (value = sum of planes) squared."""
    name: str
    x: Tensor            # [.., planes * c]
    c: int
    planes: int
    dtype: int
    sq: Tensor           # [1, rows]

    def run(self) -> None:
        L.pixel_sqsum(self.x, self.sq.numel(), self.c, self.planes, self.c, self.planes * self.c, self.dtype, self.sq)


# ---------------------------------------------------------------------------------------------------------------------
# Fused DenseNet plan (engine/densenet.py; kernels: csrc/bcosk_dense.cu)
# ---------------------------------------------------------------------------------------------------------------------
@dataclass
class DenseBnReluFwdOp:
    """t = relu(F[:, :c] * alpha): dense plane rows + sum t^2 per pixel + ReLU bits."""
    name: str
    x: Tensor            # block feature tensor [nb, h, w, planes * c_total]
    c: int
    planes: int
    alpha: Tensor        # [c] fp32
    relu: bool
    y: Tensor            # [nb, h, w, planes * c]
    sq: Optional[Tensor]
    maskbits: Optional[Tensor]   # [rows, c/32] int32
    dtype: int

    def run(self) -> None:
        ld = self.x.shape[-1]
        L.dense_bn_relu_fwd(self.x, self.y.numel() // self.y.shape[-1], self.c, self.planes, ld, ld // self.planes, self.alpha, self.relu,
                            self.y, self.sq, self.maskbits, self.dtype)


@dataclass
class DenseBnReluBwdOp:
    """G[:, :c] (+)= g * alpha * mask  (G: fp32 feature-gradient tensor of the block)."""
    name: str
    g: Tensor            # [nb, h, w, c] fp32 or 16-bit
    c: int
    alpha: Tensor
    maskbits: Optional[Tensor]
    G: Tensor            # [nb, h, w, c_total] fp32
    accumulate: bool
    dtype: int

    def run(self) -> None:
        L.dense_bn_relu_bwd(self.g, self.g.numel() // self.g.shape[-1], self.c, self.alpha, self.maskbits, self.G, self.G.shape[-1],
                            self.accumulate, self.dtype)


@dataclass
class DenseSliceCastOp:
    """out (one 16-bit plane) = G[:, col0 : col0 + c] * gain * scale."""
    name: str
    G: Tensor            # [nb, h, w, c_total] fp32
    col0: int
    c: int
    gain: Optional[Tensor]   # [rows, c]
    scale: float
    out: Tensor          # [nb, h, w, c] 16-bit
    dtype: int

    def run(self) -> None:
        L.dense_slice_cast(self.G, self.G.shape[-1], self.col0, self.out.numel() // self.out.shape[-1], self.c, self.gain, self.scale,
                           self.out, self.dtype)


@dataclass
class CopyChannelsOp:
    """dst[:, pl * dst_pstride + dst_col : ... + c] = src[:, pl * c : (pl + 1) * c] for every plane (strided device copies)."""
    name: str
    src: Tensor          # [.., planes * c] dense
    c: int
    planes: int
    dst: Tensor          # [.., planes * c_total]
    dst_col: int

    def run(self) -> None:
        rows = self.src.numel() // self.src.shape[-1]
        es = self.src.element_size()
        ld_s, ld_d = self.src.shape[-1], self.dst.shape[-1]
        for pl in range(self.planes):
            L.copy_rows_2d(self.dst.data_ptr() + (pl * (ld_d // self.planes) + self.dst_col) * es, ld_d * es,
                           self.src.data_ptr() + pl * self.c * es, ld_s * es, self.c * es, rows)


# ---------------------------------------------------------------------------------------------------------------------
# Attention-pool head inside the fused CLIP plan (kernels: csrc/bcosk_head.cu)
# ---------------------------------------------------------------------------------------------------------------------
@dataclass
class SgemmOp:
    """C[i] = alpha * op(A[i]) op(B[i]), i < batch: fp32 row-major operands addressed as (tensor, element offset, row pitch, batch stride)."""
    name: str
    trans_a: bool
    trans_b: bool
    m: int
    n: int
    k: int
    a: Tensor
    a_off: int
    lda: int
    stride_a: int
    b: Tensor
    b_off: int
    ldb: int
    stride_b: int
    c: Tensor
    c_off: int
    ldc: int
    stride_c: int
    batch: int
    alpha: float = 1.0
    accumulate: bool = False     # C += alpha * op(A) op(B)

    def run(self) -> None:
        (L.sgemm_batched_acc if self.accumulate else L.sgemm_batched)(self.trans_a, self.trans_b, self.m, self.n, self.k, self.a.data_ptr() + 4 * self.a_off, self.lda, self.stride_a,
                        self.b.data_ptr() + 4 * self.b_off, self.ldb, self.stride_b, self.c.data_ptr() + 4 * self.c_off, self.ldc,
                        self.stride_c, self.batch, self.alpha)


@dataclass
class HeadTokensOp:
    name: str
    x: Tensor            # [nb, h, w, planes * c]
    c: int
    planes: int
    dtype: int
    tokens: Tensor       # [nb, h*w + 1, c] fp32

    def run(self) -> None:
        nb, h, w, _ = self.x.shape
        L.head_tokens(self.x, nb, h * w, self.c, self.planes, self.dtype, self.tokens)


@dataclass
class RowSoftmaxOp:
    name: str
    s: Tensor            # [..., n] fp32, in place

    def run(self) -> None:
        L.row_softmax(self.s, self.s.numel() // self.s.shape[-1], self.s.shape[-1])


@dataclass
class SeedFromTokensOp:
    name: str
    g_tokens: Tensor     # [nb, npix + 1, c] fp32
    scale: float
    mul1: Optional[Tensor]
    out1: Tensor         # [nb, h, w, planes * c]
    mask2: Optional[Tensor]
    mul2: Optional[Tensor]
    out2: Optional[Tensor]
    planes: int
    dtype: int

    def run(self) -> None:
        nb, t, c = self.g_tokens.shape
        L.seed_from_tokens(self.g_tokens, nb, t - 1, c, self.scale, self.mul1, self.out1, self.mask2, self.mul2, self.out2, self.planes, self.dtype)


@dataclass
class StemIm2colOp:
    """include/bcosk.h bcosk_stem_im2col_u8: uint8 image -> stem patch matrix (v_R, v_G, v_B, 1 per tap) + 1/||patch||."""
    name: str
    x: Tensor            # [nb, 3, h, w] uint8
    k: int
    stride: int
    pad: int
    mean6: Tuple[float, ...]
    inv_std6: Tuple[float, ...]
    a_scale: float
    out: Tensor          # [nb, op, oq, kp] 16-bit, one plane
    inv_norm: Tensor     # [nb*op*oq] fp32
    dtype: int

    def run(self) -> None:
        L.stem_im2col_u8(self.x, self.k, self.stride, self.pad, self.mean6, self.inv_std6, self.a_scale, self.out, self.out.shape[-1],
                         self.inv_norm, self.dtype)


def run_ops(ops) -> None:
    for o in ops:
        o.run()
