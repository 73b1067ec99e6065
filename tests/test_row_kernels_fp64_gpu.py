"""-m gpu: the bandwidth kernels between the GEMMs against an fp64 evaluation of the same operation, element by element.

Average pooling (`avgpool_fwd`, `avgpool_bwd_mul`, both kernels of each), `pixel_sqsum`, the DenseNet consumer BN + ReLU
(`dense_bn_relu_fwd` / `_bwd`, `dense_slice_cast`, `copy_rows_2d`), the ViT row kernels (`vit_ln_fwd`, `vit_ln_bwd[_full]`,
`vit_gelu_fwd`, `vit_quickgelu_fwd`) and the CLIP RN attention-pool head (`sgemm_batched`, `head_tokens`, `row_softmax`).
tests/test_kernels_gpu.py and the model tests compare them with the fp32 emulator at toy shapes under one flat tolerance; here
every reference is fp64, computed from the exact operands the kernel reads (16-bit planes, fp32 multipliers, host scalars after
rounding to fp32), geometries are collected from the plans (tests/opsutil.py) plus the branches no plan reaches, and every element
has its own bound derived from the kernel's order of operations. With u = 2^-24 (the build has no fast-math, FMA contraction is
on; every bound holds with or without it):

* fp32 roundings: a sum of n terms costs (n - 1) u of the sum of |terms| (a sequential chain of m terms per lane followed by a
  shuffle tree of L levels: (m - 1 + L) u); an addition to 0 is exact; products, quotients, sqrtf u each; erff and expf within
  2 ulp (4 u of the value); sqrt.approx.ftz taken as 2^-22 relative.
* a tap's value is the fp32 sum of its planes: exact when the planes span <= 24 significant bits, otherwise one rounding per
  plane after the first: (planes - 1) u of the value.
* storage in P 16-bit planes: 2^-11P (fp16) / 2^-8P (bf16) of the value, plus half the fp16 subnormal spacing per plane; every
  later plane is the round-to-nearest residual of the planes before it (`check_residual_planes`).
* sums of squares (`sq`) are taken over the STORED values (include/bcosk.h): bounded by the fp32 sum alone, far below a storage
  rounding, so a kernel that squared the unrounded values fails.
* decisions (ReLU bits) must match the fp64 decision wherever the fp64 value lies farther from 0 than its bound.

Negative controls feed numerical variants of the references (count_include_pad=False pooling, sq over the unrounded values, a
one-pass LayerNorm variance, one plane where the launch writes two) to the same checkers, which must reject them.  Every case
prints its largest error as a fraction of its bound (REPORT lines, `pytest -s`).  The host-side path-coverage test needs no GPU:
`pytest -m "not gpu" tests/test_row_kernels_fp64_gpu.py` runs it (`-k "not gpu"` deselects the whole module by its name).
"""
import math
import zlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import opsutil
from opsutil import check_residual_planes, joined, store_bound
from bcos_b200.engine import ops as O

U = 2.0 ** -24
DT = {"fp16": torch.float16, "bf16": torch.bfloat16}
FORMATS = [(dt, pl) for dt in ("fp16", "bf16") for pl in (1, 2, 3)]
DTYPE_CODE = {"bf16": 1, "fp16": 0}          # bcos_b200._lib.DTYPE_CODE (kept here: the CPU test does not load the library)
SQRT_APPROX = 2.0 ** -22


def _gen(name, device="cuda"):
    """generator seeded from the case name (crc32: str hashes are salted per process)"""
    return torch.Generator(device=device).manual_seed(zlib.crc32(name.encode()))


def _f32(v) -> float:
    return float(np.float32(v))


def _ratio(err, bound) -> float:
    return float((err / bound.clamp_min(1e-300)).max()) if err.numel() else 0.0


def _report(what, ratio):
    print(f"REPORT {what}: max err/bound {ratio:.3f}")
    assert ratio <= 1.0, (what, ratio)


def _reject(what, ratio):
    """a negative control: the checker must find the variant outside its bound"""
    print(f"REPORT control {what}: max err/bound {ratio:.3g} (rejected)")
    assert ratio > 1.0, (what, "the checker accepts a wrong reference", ratio)


def _planes_tensor(shape, c, planes, dtype, gen, scale=1.0, offset=0.0):
    """[..., planes * c] 16-bit: an fp32 random value split into `planes` round-to-nearest residual planes"""
    v = (torch.randn(*shape, c, device="cuda", generator=gen) * scale + offset).double()
    out, r = [], v
    for _ in range(planes):
        p = r.to(DT[dtype])
        out.append(p)
        r = r - p.double()
    return torch.cat(out, -1)


def _lib():
    from bcos_b200 import _lib as L
    return L


# =====================================================================================================================
# average pooling: host selection rules (bcosk_avgpool_fwd / bcosk_avgpool_bwd_mul, csrc/bcosk_elementwise.cu)
# =====================================================================================================================
def _lanes_per_pixel(c):
    g, lanes = c // 8, 1
    while lanes * 2 <= g and lanes * 2 <= 32:
        lanes *= 2
    return lanes


def pool_fwd_path(w, c, planes, k, op, oq):
    """("rows", split) or ("direct", KT) as bcosk_avgpool_fwd picks it; split is clamped to the output columns"""
    smem_row = k * w * planes * c * 2
    cg = c // 8
    if cg <= 32 and cg & (cg - 1) == 0 and smem_row <= 100 * 1024 and op <= 32767:
        split = 3 if smem_row > 88 * 1024 else (2 if smem_row > 44 * 1024 else 1)
        return ("rows", min(split, oq))
    return ("direct", k if k in (2, 3) else 0)


def pool_bwd_path(h, w, c, planes, k, stride, oq, gain, sqrt_scale):
    """"rows" or "direct" as bcosk_avgpool_bwd_mul picks it (gain None / "16" / "f32"); gain_sqrt_scale needs the rows kernel"""
    smem = (w + 2 * oq) * c * 2
    if planes == 1 and gain == "16" and k <= 2 * stride and smem <= 48 * 1024 and h <= 65535:
        return "rows"
    assert not sqrt_scale, "gain_sqrt_scale needs the row-staged kernel"
    return "direct"


def _out_size(n, k, s, pad):
    return (n + 2 * pad - k) // s + 1


def _pool_fwd_plan_geometries():
    """{(h, w, c, planes, k, stride, pad, op, oq): tag} of every AvgPoolFwdOp of the plans"""
    out = {}
    for tag, op in opsutil.ops_of(O.AvgPoolFwdOp):
        _, h, w, _ = op.x.shape
        out.setdefault((h, w, op.c, op.planes, op.k, op.stride, op.pad, op.y.shape[1], op.y.shape[2]), tag)
    return out


def _pool_fwd_extra():
    """branches the plans do not reach: split 2 / 3 with oq not divisible by the split and padded last rows / columns, the split
    clamp (a global pool with one output column), the direct kernel at c / 8 = 40 / 56 / 64 / 112 with KT = 2 / 3 / generic k"""
    g = [(11, 77, 64, 2, 3, 2, 1), (11, 163, 32, 3, 3, 2, 1), (9, 118, 64, 2, 3, 2, 1), (13, 13, 16, 1, 3, 2, 1),
         (7, 7, 256, 2, 7, 7, 0), (7, 7, 256, 2, 9, 9, 1)]
    g += [(14, 14, c, 1, 2, 2, 0) for c in (320, 448)] + [(15, 15, c, 2, 3, 2, 1) for c in (512, 896)]
    g += [(13, 13, 320, 3, 5, 2, 2), (9, 9, 64, 1, 7, 1, 3)]
    return {(h, w, c, pl, k, s, p, _out_size(h, k, s, p), _out_size(w, k, s, p)): "extra" for h, w, c, pl, k, s, p in g}


def pool_fwd_cases():
    geoms = dict(_pool_fwd_extra())
    geoms.update(_pool_fwd_plan_geometries())
    return sorted(geoms.items())


def _pool_bwd_plan_geometries():
    """{(h, w, c, planes, k, stride, pad, op, oq, row_pitch, img_pitch, gain, sqrt_scale): tag} of every AvgPoolBwdMulOp"""
    out = {}
    for tag, op in opsutil.ops_of(O.AvgPoolBwdMulOp):
        _, h, w, ld = op.gx.shape
        rp, ip = op.gx.stride(1) // ld, op.gx.stride(0) // ld
        gain = None if op.gain is None else ("f32" if op.gain.dtype == torch.float32 else "16")
        out.setdefault((h, w, op.c, op.planes, op.k, op.stride, op.pad, op.gy.shape[1], op.gy.shape[2], rp, ip, gain,
                        op.gain_sqrt_scale is not None), tag)
    return out


def _pool_bwd_extra():
    """gain absent / 16-bit / fp32 on both kernels, gain_sqrt_scale (ResNet / DenseNet pool.bwd in the modes that keep the ReLU
    output), pitches wider than the image, rows and columns no window covers (k < stride, and k = 2 stride - 1 with a short
    trailing row), several planes on the direct kernel"""
    g = []
    for gain in (None, "16", "f32"):
        g += [(15, 15, 64, 1, 3, 2, 1, gain, False, 3), (14, 14, 32, 1, 2, 3, 0, gain, False, 0), (13, 13, 16, 2, 1, 2, 0, gain, False, 2)]
    g += [(15, 15, 64, 1, 3, 2, 1, "16", True, 3), (13, 13, 32, 1, 2, 3, 0, "16", True, 0), (14, 14, 320, 1, 2, 2, 0, "16", True, 1)]
    g += [(14, 14, 448, 3, 2, 2, 0, "f32", False, 1), (12, 12, 64, 1, 5, 2, 2, "16", False, 0), (9, 9, 64, 2, 4, 1, 1, None, False, 1)]
    out = {}
    for h, w, c, pl, k, s, p, gain, sq, extra_pitch in g:
        op_, oq_ = _out_size(h, k, s, p), _out_size(w, k, s, p)
        rp = w + extra_pitch
        out[(h, w, c, pl, k, s, p, op_, oq_, rp, (h + extra_pitch) * rp, gain, sq)] = "extra"
    return out


def pool_bwd_cases():
    geoms = dict(_pool_bwd_extra())
    geoms.update(_pool_bwd_plan_geometries())
    return sorted(geoms.items(), key=str)


def _sgemm_plan_geometries():
    out = {}
    for tag, op in opsutil.ops_of(O.SgemmOp):
        out.setdefault((op.trans_a, op.trans_b, op.m, op.n, op.k, op.lda, op.stride_a, op.ldb, op.stride_b, op.ldc, op.stride_c,
                        op.batch, op.alpha), tag)
    return out


def _sgemm_extra():
    """(trans_a, trans_b, m, n, k, batch, alpha, pad): every transpose pair at both tile widths, ragged m / n / k, ld and batch
    strides `pad` elements wider than the row"""
    g = []
    for ta in (False, True):
        for tb in (False, True):
            g += [(ta, tb, 37, 45, 70, 3, 0.37, 5), (ta, tb, 300, 290, 83, 12, -1.5, 3)]
    g += [(False, True, 1, 1, 1, 1, 1.0, 0), (True, False, 129, 65, 17, 40, 2.0 ** -7, 1)]
    return g


def sgemm_tile_width(m, n, batch):
    """bcosk_sgemm_batched: 32 x 32 tiles below 296 tiles of 64 x 64, 64 x 64 otherwise"""
    tiles64 = ((n + 63) // 64) * ((m + 63) // 64) * batch
    return 32 if tiles64 < 2 * 148 else 64


# =====================================================================================================================
# path coverage (CPU)
# =====================================================================================================================
def test_parametrisation_reaches_every_pooling_and_sgemm_branch():
    """Restates the host selection rules of the pooling and SGEMM entry points, labels every collected geometry with the kernel it
    takes, and asserts the suite reaches the row-staged forward at splits 1 / 2 / 3 (and the clamp of the split to oq), the direct
    forward at KT = 2 / 3 / generic with c / 8 above 32 and not a power of two, both backward kernels with every gain kind, the
    gain_sqrt_scale multiplier, uncovered input rows, wider output pitches, and both SGEMM tile widths with all four transposes."""
    fwd = {}
    for (h, w, c, pl, k, s, p, op_, oq_), tag in pool_fwd_cases():
        path = pool_fwd_path(w, c, pl, k, op_, oq_)
        fwd.setdefault(path, []).append((h, w, c, pl, k, s, p, tag))
        if path[0] == "rows":
            raw = 3 if k * w * pl * c * 2 > 88 * 1024 else (2 if k * w * pl * c * 2 > 44 * 1024 else 1)
            if raw > oq_:
                fwd.setdefault("clamped", []).append((h, w, c, pl, k, s, p))
            if path[1] > 1 and oq_ % path[1]:
                fwd.setdefault(("ragged", path[1]), []).append((h, w, c, pl, k, s, p))
    for key, val in sorted(fwd.items(), key=str):
        print(f"pool fwd {key}: {len(val)} geometries, e.g. {val[0]}")
    need = [("rows", 1), ("rows", 2), ("rows", 3), ("direct", 2), ("direct", 3), ("direct", 0), "clamped", ("ragged", 2), ("ragged", 3)]
    assert all(n in fwd for n in need), [n for n in need if n not in fwd]
    direct_cg = {g[2] // 8 for key, v in fwd.items() if isinstance(key, tuple) and key[0] == "direct" for g in v}
    assert {40, 56, 64, 112} <= direct_cg, direct_cg
    assert {g[3] for v in fwd.values() for g in v} == {1, 2, 3}
    assert any(t != "extra" for v in fwd.values() for *_, t in v if isinstance(t, str))

    bwd = {}
    for (h, w, c, pl, k, s, p, op_, oq_, rp, ip, gain, sq), tag in pool_bwd_cases():
        path = pool_bwd_path(h, w, c, pl, k, s, oq_, gain, sq)
        bwd.setdefault((path, gain), []).append(tag)
        if sq:
            bwd.setdefault("sqrt_scale", []).append(tag)
        if rp > w or ip > h * rp:
            bwd.setdefault(("pitch", path), []).append(tag)
        covered = set()
        for q in range(op_):
            covered.update(range(q * s - p, q * s - p + k))
        if set(range(h)) - covered:
            bwd.setdefault(("uncovered", path), []).append(tag)
    print("pool bwd:", {str(k): len(v) for k, v in bwd.items()})
    need = [("rows", "16"), ("direct", None), ("direct", "16"), ("direct", "f32"), "sqrt_scale", ("pitch", "rows"),
            ("pitch", "direct"), ("uncovered", "rows"), ("uncovered", "direct")]
    assert all(n in bwd for n in need), [n for n in need if n not in bwd]

    widths = {}
    for ta, tb, m, n, k, batch, alpha, pad in _sgemm_extra():
        widths.setdefault(sgemm_tile_width(m, n, batch), set()).add((ta, tb))
    for key, tag in _sgemm_plan_geometries().items():
        widths.setdefault(sgemm_tile_width(key[2], key[3], key[11]), set()).add((key[0], key[1]))
    print("sgemm tile widths:", widths)
    every = {(a, b) for a in (False, True) for b in (False, True)}
    assert widths.get(32, set()) >= every and widths.get(64, set()) >= every, widths
    assert _sgemm_plan_geometries(), "the CLIP RN fused head launches no SGEMM any more"


# =====================================================================================================================
# average pooling forward
# =====================================================================================================================
def _nchw(t):
    return t.permute(0, 3, 1, 2)


def _pool_fwd_reference(xj, k, s, p, op_, oq_, include_pad=True):
    """fp64 pooled value [nb, op, oq, c] and the mean of |tap| (the fp32 sum's bound is a multiple of it)"""
    ref = F.avg_pool2d(_nchw(xj), k, s, p, count_include_pad=include_pad)[:, :, :op_, :oq_]
    a = F.avg_pool2d(_nchw(xj.abs()), k, s, p, count_include_pad=True)[:, :, :op_, :oq_]
    return ref.permute(0, 2, 3, 1), a.permute(0, 2, 3, 1)


def _pool_fwd_check(y, sq, ref, a, dtype, planes, c, k, what):
    """(value ratio, sq ratio): fp32 tap sums of <= k^2 taps ((planes - 1) u per tap), * fl(1/k^2), storage; sq over the stored
    values: a chain of 8 ceil(c / 8 / lanes) fma per lane, log2(lanes) shuffle levels, 2 (planes - 1) u for the stored fp32 value"""
    e = (planes + k * k) * U * a
    got = joined(y, planes, c)
    rv = _ratio((got - ref).abs(), store_bound(ref, e, dtype, planes))
    rs = 0.0
    if sq is not None:
        lanes = _lanes_per_pixel(c)
        depth = 8 * -(-(c // 8) // lanes) + int(math.log2(lanes)) + 2 * (planes - 1)
        sq64 = (got * got).sum(-1)
        rs = _ratio((sq.view(sq64.shape).double() - sq64).abs(), depth * U * sq64)
    return rv, rs


@pytest.mark.gpu
@pytest.mark.parametrize("geom,tag", pool_fwd_cases(), ids=lambda v: "x".join(map(str, v)) if isinstance(v, tuple) else v)
def test_avgpool_fwd_within_fp64_bound(bcosk_lib, geom, tag):
    """avgpool_fwd at every plan geometry and the extra branches, six formats, batch 2: values within their bound, planes =
    residuals, sq = the sum of the STORED values squared; sq = None writes the same y.  Controls: count_include_pad=False at the
    border, sq over the unrounded values, one plane of a two-plane store."""
    L = _lib()
    h, w, c, planes, k, s, p, op_, oq_ = geom
    nb = 2
    path = pool_fwd_path(w, c, planes, k, op_, oq_)
    worst = []
    for dtype, pl in FORMATS:
        gen = _gen(f"poolf{geom}{dtype}{pl}")
        x = _planes_tensor((nb, h, w), c, pl, dtype, gen)
        y = torch.full((nb, op_, oq_, pl * c), float("nan"), dtype=DT[dtype], device="cuda")
        sq = torch.full((nb * op_ * oq_,), float("nan"), device="cuda")
        L.avgpool_fwd(x, nb, h, w, c, pl, k, s, p, y, op_, oq_, DTYPE_CODE[dtype], sq)
        y2 = torch.full_like(y, float("nan"))
        L.avgpool_fwd(x, nb, h, w, c, pl, k, s, p, y2, op_, oq_, DTYPE_CODE[dtype], None)
        torch.cuda.synchronize()
        what = f"avgpool_fwd {geom} {dtype}x{pl} {path}"
        assert torch.equal(y.view(torch.int16), y2.view(torch.int16)), (what, "sq = None changes y")
        check_residual_planes(y, pl, c, what)
        xj = joined(x, pl, c)
        ref, a = _pool_fwd_reference(xj, k, s, p, op_, oq_)
        rv, rs = _pool_fwd_check(y, sq, ref, a, dtype, pl, c, k, what)
        worst.append(f"{dtype}x{pl} {rv:.3f}/{rs:.3f}")
        assert rv <= 1.0 and rs <= 1.0, (what, rv, rs)
        if pl == 1 and dtype == "bf16":
            if p > 0:
                bad, _ = _pool_fwd_reference(xj, k, s, p, op_, oq_, include_pad=False)
                _reject(f"avgpool_fwd {geom} count_include_pad=False", _pool_fwd_check(y, None, bad, a, dtype, pl, c, k, what)[0])
            sq_bad = (ref * ref).sum(-1).float()
            _reject(f"avgpool_fwd {geom} sq of the unrounded values", _pool_fwd_check(y, sq_bad, ref, a, dtype, pl, c, k, what)[1])
        if pl == 2 and dtype == "fp16":
            _reject(f"avgpool_fwd {geom} one plane of two",
                    _pool_fwd_check(torch.cat([y[..., :c], torch.zeros_like(y[..., :c])], -1), None, ref, a, dtype, pl, c, k, what)[0])
    print(f"REPORT avgpool_fwd {'x'.join(map(str, geom))} nb={nb} {path} ({tag}): value / sq max err/bound " + " ".join(worst))


# =====================================================================================================================
# average pooling backward (x gain)
# =====================================================================================================================
@pytest.mark.gpu
@pytest.mark.parametrize("geom,tag", pool_bwd_cases(), ids=lambda v: "x".join(map(str, v)) if isinstance(v, tuple) else v)
def test_avgpool_bwd_mul_within_fp64_bound(bcosk_lib, geom, tag):
    """avgpool_bwd_mul: gx = gain (or sqrt(gain * scale)) * sum of the covering output gradients / k^2, written through the launch's
    row / image pitch.  Bound: (planes - 1 + taps - 1) u of sum |taps|, fl(1/k^2 * gain) and the product (+ 0.5 u + 2^-22 through
    the approximate sqrt), storage.  Input pixels no window covers are exactly 0; pixels outside the view keep their NaN."""
    L = _lib()
    h, w, c, planes, k, s, p, op_, oq_, rp, ip, gain_kind, use_sqrt = geom
    nb = 2
    path = pool_bwd_path(h, w, c, planes, k, s, oq_, gain_kind, use_sqrt)
    fmts = [(dt, planes) for dt in ("fp16", "bf16")]
    worst = []
    for dtype, pl in fmts:
        gen = _gen(f"poolb{geom}{dtype}")
        gy = _planes_tensor((nb, op_, oq_), c, pl, dtype, gen)
        gain = None
        if gain_kind is not None:
            g32 = torch.rand(nb * h * w, c, device="cuda", generator=gen) * 2 + 0.01
            gain = g32 if gain_kind == "f32" else g32.to(DT[dtype])
        scale = torch.rand(nb * h * w, device="cuda", generator=gen) * 3 + 0.05 if use_sqrt else None
        ld = pl * c
        buf = torch.full((nb * ip * ld,), float("nan"), dtype=DT[dtype], device="cuda")
        gx = buf.as_strided((nb, h, w, ld), (ip * ld, rp * ld, ld, 1))
        L.avgpool_bwd_mul(gy, nb, h, w, c, pl, k, s, p, op_, oq_, gain, gain_kind == "f32", gx, DTYPE_CODE[dtype], scale)
        torch.cuda.synchronize()
        what = f"avgpool_bwd_mul {geom} {dtype}x{pl} {path}"
        inside = torch.zeros(buf.numel(), dtype=torch.bool, device="cuda")
        inside.as_strided(gx.shape, gx.stride()).fill_(True)
        assert torch.isnan(buf[~inside].float()).all(), (what, "wrote outside the view")
        gxc = gx.contiguous()
        check_residual_planes(gxc, pl, c, what)
        gyj = _nchw(joined(gy, pl, c))
        ones = torch.ones(1, 1, k, k, dtype=torch.float64, device="cuda")
        wgt = ones.expand(c, 1, k, k)

        def spread(t):        # sum over the windows covering each input pixel (adjoint of the window sum)
            o = F.conv_transpose2d(t, wgt, stride=s, groups=c)           # index j = input pixel j - pad
            full = torch.zeros(nb, c, max(h + p, o.shape[2]), max(w + p, o.shape[3]), dtype=torch.float64, device="cuda")
            full[:, :, :o.shape[2], :o.shape[3]] = o
            return full[:, :, p:p + h, p:p + w].permute(0, 2, 3, 1)
        S, A = spread(gyj), spread(gyj.abs())
        cover = spread(torch.ones_like(gyj))
        taps = cover.clamp_min(1)
        m64 = torch.full_like(S, 1.0 / (k * k))
        rel_m = 2 * U
        if gain is not None:
            gv = gain.double().view(nb, h, w, c)
            if use_sqrt:
                gv = (gv * scale.double().view(nb, h, w, 1)).sqrt()
                rel_m += 0.5 * U + SQRT_APPROX
            m64 = m64 * gv
        ref = S * m64
        e = (pl - 1 + taps - 1) * U * A * m64.abs() + rel_m * (S * m64).abs() + U * ref.abs()
        got = joined(gxc, pl, c)
        unc = cover == 0
        assert torch.equal(got[unc], torch.zeros_like(got[unc])), (what, "an input pixel no window covers is not 0")
        r = _ratio((got - ref).abs(), store_bound(ref, e, dtype, pl))
        worst.append(f"{dtype}x{pl} {r:.3f}")
        assert r <= 1.0, (what, r)
    print(f"REPORT avgpool_bwd_mul {'x'.join(map(str, geom))} nb={nb} {path} ({tag}, {int(unc[0, ..., 0].sum())} uncovered pixels): "
          f"max err/bound " + " ".join(worst))


# =====================================================================================================================
# pixel_sqsum
# =====================================================================================================================
@pytest.mark.gpu
@pytest.mark.parametrize("c,extra", [(64, 0), (256, 16), (1024, 8), (2048, 0), (200, 24)])
def test_pixel_sqsum_within_fp64_bound(bcosk_lib, c, extra):
    """pixel_sqsum over the six formats with a plane stride `extra` columns wider than c (and the row pitch wider again): the sum
    of the joined planes squared, 8 ceil(c / 256) fma per lane + 5 shuffle levels + 2 (planes - 1) u for the fp32 tap value."""
    L = _lib()
    rows = 1000
    worst = []
    for dtype, pl in FORMATS:
        gen = _gen(f"sqsum{c}{extra}{dtype}{pl}")
        ps = c + extra
        ld = pl * ps + 8 * (extra > 0)
        x = torch.full((rows, ld), float("nan"), dtype=DT[dtype], device="cuda")
        v = _planes_tensor((rows,), c, pl, dtype, gen)
        for i in range(pl):
            x[:, i * ps:i * ps + c] = v[:, i * c:(i + 1) * c]
        sq = torch.full((rows,), float("nan"), device="cuda")
        L.pixel_sqsum(x, rows, c, pl, ps, ld, DTYPE_CODE[dtype], sq)
        torch.cuda.synchronize()
        xj = joined(v, pl, c)
        sq64 = (xj * xj).sum(-1)
        depth = 8 * -(-c // 256) + 5 + 2 * (pl - 1)
        r = _ratio((sq.double() - sq64).abs(), depth * U * sq64)
        worst.append(f"{dtype}x{pl} {r:.3f}")
        assert r <= 1.0, (c, extra, dtype, pl, r)
    print(f"REPORT pixel_sqsum c={c} plane_stride=c+{extra} rows={rows}: max err/bound " + " ".join(worst))


# =====================================================================================================================
# DenseNet consumer BN + ReLU
# =====================================================================================================================
def _dense_channel_counts():
    cs = {op.c for _, op in opsutil.ops_of(O.DenseBnReluFwdOp)}
    return sorted(cs)


def _mask_dense(mask, c):
    m = mask.long() & 0xffffffff
    ch = torch.arange(c, device=mask.device)
    return ((m[:, ch // 32] >> (ch % 32)) & 1).bool()


@pytest.mark.gpu
def test_dense_bn_relu_fwd_bwd_within_fp64_bound(bcosk_lib):
    """dense_bn_relu_fwd at every consumer channel count of the DenseNet plans (64 + 32 j) plus c = 200 (c % 32 != 0: no mask bits,
    which the host refuses there) from a feature tensor whose plane stride is wider than c, six formats, relu on / off: t = f alpha
    (planes - 1 + 1) u, storage, sq, and the ReLU bits equal to the fp64 decision wherever |f alpha| exceeds its bound.  Then
    dense_bn_relu_bwd on the same bits: G = (G | 0) + g alpha mask with g fp32 / 16-bit, accumulate 0 / 1, mask absent / present;
    columns >= c of G untouched."""
    L = _lib()
    cs = _dense_channel_counts()
    assert len(cs) >= 10 and min(cs) == 64 and all(c % 32 == 0 for c in cs), cs
    rows = 96
    worst = {"y": 0.0, "sq": 0.0, "G": 0.0}
    nbits = 0
    for c in cs + [200]:
        for dtype, pl in FORMATS:
            for relu in (True, False):
                gen = _gen(f"dense{c}{dtype}{pl}{relu}")
                pstride = c + 48
                F16 = _planes_tensor((rows,), pstride, pl, dtype, gen)
                alpha = torch.randn(c, device="cuda", generator=gen)
                alpha[::7] = 0.0
                y = torch.full((rows, pl * c), float("nan"), dtype=DT[dtype], device="cuda")
                sq = torch.full((rows,), float("nan"), device="cuda")
                words = (c + 31) // 32
                # prefilled with the complement of what relu = False must write: a word the kernel skips fails either way
                mask = torch.full((rows, words), -1 if relu else 0, dtype=torch.int32, device="cuda") if c % 32 == 0 else None
                L.dense_bn_relu_fwd(F16, rows, c, pl, pl * pstride, pstride, alpha, relu, y, sq, mask, DTYPE_CODE[dtype])
                torch.cuda.synchronize()
                what = f"dense_bn_relu_fwd c={c} {dtype}x{pl} relu={relu}"
                fj = sum(F16[:, i * pstride:i * pstride + c].double() for i in range(pl))
                t64 = fj * alpha.double()
                e = pl * U * t64.abs()
                ref = t64.clamp_min(0) if relu else t64
                check_residual_planes(y, pl, c, what)
                got = joined(y, pl, c)
                clear = t64.abs() > e
                if relu:
                    # near-0 values may fall either way: compare them with the value the decision picked
                    ref = torch.where(clear, ref, torch.where(got == 0, torch.zeros_like(ref), t64))
                r = _ratio((got - ref).abs(), store_bound(ref, e, dtype, pl))
                sq64 = (got * got).sum(-1)
                depth = 8 * -(-(c // 8) // 32) + 5 + 2 * (pl - 1)
                rs = _ratio((sq.double() - sq64).abs(), depth * U * sq64)
                assert r <= 1.0 and rs <= 1.0, (what, r, rs)
                worst["y"], worst["sq"] = max(worst["y"], r), max(worst["sq"], rs)
                if mask is not None:
                    md = _mask_dense(mask, c)
                    want = (t64 > 0) if relu else torch.ones_like(clear)
                    assert torch.equal(md[clear], want[clear]), (what, "ReLU bits differ from the fp64 decision")
                    assert md[got != 0].all(), (what, "a stored non-zero value without its bit")
                    if not relu:
                        assert (mask == -1).all(), (what, "relu = False must set every bit of every word")
                    nbits += int(clear.sum())
                else:
                    with pytest.raises(RuntimeError):
                        L.dense_bn_relu_fwd(F16, rows, c, pl, pl * pstride, pstride, alpha, relu, y, sq,
                                            torch.zeros(rows, words, dtype=torch.int32, device="cuda"), DTYPE_CODE[dtype])
                if pl != 1 or not relu:
                    continue
                # backward through the same bits
                g_ld = c + 24
                for gk in ("f32", "16"):
                    for acc in (False, True):
                        for use_mask in ((False, True) if mask is not None else (False,)):
                            g32 = torch.randn(rows, c, device="cuda", generator=gen)
                            g = g32 if gk == "f32" else g32.to(DT[dtype])
                            G0 = torch.randn(rows, g_ld, device="cuda", generator=gen)
                            G = G0.clone()
                            L.dense_bn_relu_bwd(g, rows, c, alpha, mask if use_mask else None, G, g_ld, acc, DTYPE_CODE[dtype])
                            torch.cuda.synchronize()
                            wb = f"dense_bn_relu_bwd c={c} {dtype} g={gk} accumulate={acc} mask={use_mask}"
                            assert torch.equal(G[:, c:], G0[:, c:]), (wb, "columns >= c changed")
                            md = _mask_dense(mask, c) if use_mask else torch.ones(rows, c, dtype=torch.bool, device="cuda")
                            prod = g.double() * alpha.double() * md
                            base = G0[:, :c].double() if acc else 0.0
                            ref_g = base + prod
                            rg = _ratio((G[:, :c].double() - ref_g).abs(), U * prod.abs() + U * ref_g.abs())
                            assert rg <= 1.0, (wb, rg)
                            worst["G"] = max(worst["G"], rg)
    print(f"REPORT dense_bn_relu_fwd / _bwd c in {cs + [200]} (six formats, relu on / off; bwd: g fp32 / 16-bit, accumulate, mask; "
          f"{nbits} decided ReLU bits): max err/bound y {worst['y']:.3f} sq {worst['sq']:.3f} G {worst['G']:.3f}")


@pytest.mark.gpu
def test_dense_slice_cast_and_copy_rows(bcosk_lib):
    """dense_slice_cast: out (one plane) = fl(fl(G[:, col0:col0 + c] gain) scale), gain absent / 16-bit / fp32, col0 > 0, scale != 1:
    2 u + storage.  copy_rows_2d through every CopyChannelsOp geometry of the plans: bit-exact, bytes outside the slice unchanged."""
    L = _lib()
    rows, worst = 300, 0.0
    for dtype in ("fp16", "bf16"):
        for c, col0, g_ld in ((64, 32, 256), (128, 4, 200), (448, 64, 512)):
            for gk in (None, "16", "f32"):
                for scale in (1.0, 0.3, 1024.0):
                    gen = _gen(f"slice{dtype}{c}{col0}{gk}{scale}")
                    G = torch.randn(rows, g_ld, device="cuda", generator=gen)
                    gain = None
                    if gk is not None:
                        g32 = torch.rand(rows, c, device="cuda", generator=gen) * 2
                        gain = g32 if gk == "f32" else g32.to(DT[dtype])
                    out = torch.full((rows, c), float("nan"), dtype=DT[dtype], device="cuda")
                    L.dense_slice_cast(G, g_ld, col0, rows, c, gain, scale, out, DTYPE_CODE[dtype])
                    torch.cuda.synchronize()
                    ref = G[:, col0:col0 + c].double() * (gain.double() if gain is not None else 1.0) * _f32(scale)
                    e = (2 if gain is not None else 1) * U * ref.abs()
                    r = _ratio((out.double() - ref).abs(), store_bound(ref, e, dtype, 1))
                    assert r <= 1.0, (dtype, c, col0, gk, scale, r)
                    worst = max(worst, r)
    # copy_rows_2d: the input of every dense block (the pooled transition output, `planes` planes of c_in channels) goes to channels
    # [0, c_in) of every plane of the block's feature tensor, whose plane stride is the block's c_total (DENSENET_ARCH: c_in + growth
    # x layers; a transition halves the channels) - stated here from the architecture, not from the launch record
    from bcos_b200.engine.densenet import DENSENET_ARCH
    seen = set()
    for tag, op in opsutil.ops_of(O.CopyChannelsOp):
        arch = tag.split("/")[-1].split("@")[0]
        bi = int(op.name.split(".")[0][len("denseblock"):])
        growth, blocks, c_in = DENSENET_ARCH[arch]
        for n in blocks[:bi - 1]:
            c_in = (c_in + growth * n) // 2
        c_total = c_in + growth * blocks[bi - 1]
        key = (arch, bi, op.planes)
        if key in seen:
            continue
        seen.add(key)
        what = f"copy_rows_2d {tag} {op.name} planes={op.planes} c_in={c_in} c_total={c_total}"
        assert op.c == c_in and op.dst_col == 0 and op.dst.shape[-1] == op.planes * c_total, what
        pix = op.src.numel() // op.src.shape[-1]
        gen = _gen(f"copy{key}")
        src = torch.randn(pix, op.planes * c_in, device="cuda", generator=gen).to(op.src.dtype)
        dst = torch.randn(pix, op.planes * c_total, device="cuda", generator=gen).to(op.dst.dtype)
        before = dst.clone()
        O.CopyChannelsOp("copy", src, c_in, op.planes, dst, 0).run()
        torch.cuda.synchronize()
        bits = torch.int16 if dst.element_size() == 2 else torch.int32
        d3, b3 = dst.view(pix, op.planes, c_total).view(bits), before.view(pix, op.planes, c_total).view(bits)
        assert torch.equal(d3[..., :c_in], src.view(pix, op.planes, c_in).view(bits)), (what, "block input not copied bit for bit")
        assert torch.equal(d3[..., c_in:], b3[..., c_in:]), (what, "channels past the block input changed")
    assert len(seen) >= 6, seen
    _report(f"dense_slice_cast (gain none / 16-bit / fp32, col0 > 0, scale 1 / 0.3 / 1024); copy_rows_2d bit-exact at {len(seen)} "
            f"dense-block inputs of the plans", worst)


# =====================================================================================================================
# ViT LayerNorm forward
# =====================================================================================================================
def _ln_geometries():
    out = {}
    for tag, op in opsutil.ops_of(O.VitLnFwdOp):
        out.setdefault((op.d, op.planes, op.out_planes or op.planes), tag)
    return out


def _ln_reference(xj, w, eps, pl, nvec):
    """fp64 y, rstd and their bounds, following the kernel: per lane a chain of 8 ceil(nvec / 32) terms, 5 shuffle levels; the
    mean is s / d; centred values, their squares summed (two passes), var / d, rstd = 1 / sqrtf(var + eps), y = (f - mean) rstd w"""
    d = xj.shape[-1]
    depth = 8 * -(-nvec // 32) - 1 + 5
    ef = (pl - 1) * U * xj.abs()                              # the fp32 tap value
    mean = xj.mean(-1, keepdim=True)
    em = (ef.sum(-1, keepdim=True) + depth * U * (xj.abs() + ef).sum(-1, keepdim=True)) / d + U * mean.abs()
    D = xj - mean
    dl = ef + em + U * (D.abs() + ef + em)                    # fl(f - mean)
    var = (D * D).mean(-1, keepdim=True)
    evar = ((2 * D.abs() * dl + dl * dl).sum(-1, keepdim=True) + (depth + 1) * U * ((D.abs() + dl) ** 2).sum(-1, keepdim=True)) / d \
        + U * var
    ve = var + eps
    rv = (evar + U * (ve + evar)) / ve
    rel_rstd = 0.5 * rv / (1 - rv) + 2 * U
    rstd = 1.0 / ve.sqrt()
    y = D * rstd * w
    ey = (dl * rstd + D.abs() * rstd * rel_rstd) * w.abs() + 2 * U * y.abs()
    return y, ey, rstd[..., 0], (rstd * rel_rstd)[..., 0]


@pytest.mark.gpu
def test_vit_ln_fwd_within_fp64_bound(bcosk_lib):
    """vit_ln_fwd at the plans' (d, planes, out_planes) and d = 192 .. 1024 (LN_MAXV), out_planes != planes, six formats; half the
    rows have a mean 1e3 times their spread (a one-pass E[x^2] - mean^2 variance fails there: negative control).  y, rstd and sq
    (sum of the stored y squared) within their bounds."""
    L = _lib()
    geoms = dict(_ln_geometries())
    assert geoms
    for d in (192, 264, 512, 768, 1024):
        for pl, opl in ((1, 2), (3, 1), (2, 3)):
            geoms.setdefault((d, pl, opl), "extra")
    rows, eps = 64, 1e-5
    for (d, _pl, opl), tag in sorted(geoms.items()):
        worst = []
        for dtype, pl in FORMATS:
            gen = _gen(f"ln{d}{pl}{opl}{dtype}")
            # far rows: mean / std ~ 1e3 (one bf16 plane cannot resolve the spread there: those rows stay centred)
            far = torch.zeros(rows, 1, device="cuda")
            if not (dtype == "bf16" and pl == 1):
                far[rows // 2:] = 1e3
            base = torch.randn(rows, d, device="cuda", generator=gen).double() * (1 + 3 * torch.rand(rows, 1, device="cuda", generator=gen)).double()
            v = base + far.double() * (base.std(-1, keepdim=True))
            parts, r_ = [], v
            for _ in range(pl):
                q = r_.to(DT[dtype])
                parts.append(q)
                r_ = r_ - q.double()
            x = torch.cat(parts, -1)
            w = torch.randn(d, device="cuda", generator=gen)
            y = torch.full((rows, opl * d), float("nan"), dtype=DT[dtype], device="cuda")
            rstd = torch.full((rows,), float("nan"), device="cuda")
            sq = torch.full((rows,), float("nan"), device="cuda")
            L.vit_ln_fwd(x, rows, d, pl, w, eps, y, rstd, sq, DTYPE_CODE[dtype], opl)
            torch.cuda.synchronize()
            what = f"vit_ln_fwd d={d} {dtype}x{pl}->{opl}"
            xj = joined(x, pl, d)
            ref, ey, r64, er = _ln_reference(xj, w.double(), _f32(eps), pl, d // 8)
            check_residual_planes(y, opl, d, what)
            got = joined(y, opl, d)
            ry = _ratio((got - ref).abs(), store_bound(ref, ey, dtype, opl))
            rr = _ratio((rstd.double() - r64).abs(), er)
            sq64 = (got * got).sum(-1)
            rs = _ratio((sq.double() - sq64).abs(), (8 * -(-(d // 8) // 32) + 5 + 2 * (opl - 1)) * U * sq64)
            worst.append(f"{dtype}x{pl} {ry:.3f}/{rr:.3f}/{rs:.3f}")
            assert ry <= 1.0 and rr <= 1.0 and rs <= 1.0, (what, ry, rr, rs)
            if dtype == "fp16" and pl == 2:
                # one-pass variance in fp32 on the far-from-zero rows
                x32 = xj.float()
                m32 = x32.mean(-1, keepdim=True)
                var1 = ((x32 * x32).mean(-1, keepdim=True) - m32 * m32).clamp_min(0)
                bad = ((x32 - m32) / (var1 + _f32(eps)).sqrt() * w).double()
                _reject(f"vit_ln_fwd d={d} one-pass variance", _ratio((bad - ref).abs()[rows // 2:], ey[rows // 2:]))
        print(f"REPORT vit_ln_fwd d={d} out_planes={opl} rows={rows} ({tag}): y / rstd / sq max err/bound " + " ".join(worst))


# =====================================================================================================================
# ViT LayerNorm backward (explanation form, and the true form of CLIP's LayerNorm)
# =====================================================================================================================
def _ln_bwd_geometries():
    """{(d, full, x_planes): tag} of every VitLnBwdOp of the plans"""
    out = {}
    for tag, op in opsutil.ops_of(O.VitLnBwdOp):
        out.setdefault((op.d, op.x is not None, op.x_planes if op.x is not None else 0), tag)
    return out


def _row_mean(p, ep, depth):
    """fp64 mean over the last axis of terms p (each within ep of its fp32 value) and the bound of the kernel's fp32 mean:
    the lane chains and shuffle tree (depth roundings), then / d"""
    d = p.shape[-1]
    m = p.mean(-1, keepdim=True)
    return m, (ep.sum(-1, keepdim=True) + depth * U * (p.abs() + ep).sum(-1, keepdim=True)) / d + U * (m.abs() + depth * U * p.abs().mean(-1, keepdim=True))


def _ln_bwd_reference(g, w, r, G_in, xj, x_planes):
    """fp64 o = G_in + r (g w - mean(g w) [- xh mean(g w xh)]), xh = (x - mean x) r, and the bound of the kernel's fp32 evaluation:
    fl(g w), the means (lane chains + 5 shuffle levels, / d), fl(f - mean) and fl(x - mean_x) fl(* r), the fma chain of g w xh,
    fl(xh mean_gx), the subtraction, fl(* r), fl(+ G_in)"""
    d = g.shape[-1]
    depth = 8 * -(-(d // 8) // 32) - 1 + 5
    p = g * w
    ep = U * p.abs()
    mg, emg = _row_mean(p, ep, depth)
    a = p - mg
    ea = ep + emg + U * (a.abs() + ep + emg)
    if xj is not None:
        ex = (x_planes - 1) * U * xj.abs()
        mx, emx = _row_mean(xj, ex, depth)
        dx = xj - mx
        edx = ex + emx + U * (dx.abs() + ex + emx)
        xh = dx * r
        exh = r.abs() * edx + U * (xh.abs() + r.abs() * edx)
        pg = p * xh
        epg = ep * xh.abs() + (p.abs() + ep) * exh
        mgx, emgx = _row_mean(pg, epg, depth + 1)                  # fma from 0 rounds too
        t = xh * mgx
        et = xh.abs() * emgx + exh * (mgx.abs() + emgx) + U * (t.abs() + xh.abs() * emgx + exh * (mgx.abs() + emgx))
        a = a - t
        ea = ea + et + U * (a.abs() + ea + et)
    o = r * a
    eo = r.abs() * ea + U * (o.abs() + r.abs() * ea)
    if G_in is not None:
        o = o + G_in
        eo = eo + U * (o.abs() + eo)
    return o, eo


LN_BWD_OUTS = [(True, True), (True, False), (False, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("full", [False, True], ids=["vit_ln_bwd", "vit_ln_bwd_full"])
def test_vit_ln_bwd_within_fp64_bound(bcosk_lib, full):
    """vit_ln_bwd (variance detached: G_out = G_in + rstd (g w - mean(g w))) and vit_ln_bwd_full (nothing detached: x-hat recomputed from
    the x planes with the given rstd, minus xh mean(g w xh)) at the plans' d and d = 264 / 512 / 1024 (LN_MAXV), fp16 / bf16, over
    g fp32 / 16-bit, G_in absent / present, (G_out, ghat) both or either, gain absent / 16-bit / fp32 (ghat = G_out gain, one plane),
    x in 1 / 2 / 3 planes for the full form: G_out within its fp32 bound, ghat within that bound times the gain plus one rounding and the
    one-plane store."""
    L = _lib()
    geoms = {k: t for k, t in _ln_bwd_geometries().items() if k[1] == full}
    assert geoms, "no plan launches this form"
    ds = sorted({k[0] for k in geoms} | {264, 512, 1024})
    rows = 64
    for d in ds:
        tag = ", ".join(sorted({t for k, t in geoms.items() if k[0] == d})) or "extra"
        worst, n = {"G_out": 0.0, "ghat": 0.0}, 0
        for dtype in ("fp16", "bf16"):
            for xp in ((1, 2, 3) if full else (0,)):
                gen = _gen(f"lnbwd{full}{d}{dtype}{xp}")
                w = torch.randn(d, device="cuda", generator=gen)
                g32 = torch.randn(rows, d, device="cuda", generator=gen)
                G_in32 = torch.randn(rows, d, device="cuda", generator=gen)
                gain32 = torch.rand(rows, d, device="cuda", generator=gen) * 2 + 0.01
                x = xj = None
                if full:
                    v = torch.randn(rows, d, device="cuda", generator=gen) * 2 + torch.randn(rows, 1, device="cuda", generator=gen) * 3
                    parts, r_ = [], v.double()
                    for _ in range(xp):
                        q = r_.to(DT[dtype])
                        parts.append(q)
                        r_ = r_ - q.double()
                    x = torch.cat(parts, -1)
                    xj = joined(x, xp, d)
                    rstd = (1.0 / (xj.var(-1, unbiased=False) + 1e-5).sqrt()).float()
                else:
                    rstd = torch.rand(rows, device="cuda", generator=gen) * 3 + 0.1
                for gk in ("f32", "16"):
                    g = g32 if gk == "f32" else g32.to(DT[dtype])
                    for use_in in (False, True):
                        G_in = G_in32 if use_in else None
                        ref, e = _ln_bwd_reference(g.double(), w.double()[None], rstd.double()[:, None],
                                                   G_in.double() if use_in else None, xj, xp)
                        for want_out, want_hat in LN_BWD_OUTS:
                            for gnk in ((None, "16", "f32") if want_hat else (None,)):
                                gain = None if gnk is None else (gain32 if gnk == "f32" else gain32.to(DT[dtype]))
                                G_out = torch.full((rows, d), float("nan"), device="cuda") if want_out else None
                                ghat = torch.full((rows, d), float("nan"), dtype=DT[dtype], device="cuda") if want_hat else None
                                if full:
                                    L.vit_ln_bwd_full(g, x, xp, G_in, rows, d, w, rstd, G_out, gain, ghat, DTYPE_CODE[dtype])
                                else:
                                    L.vit_ln_bwd(g, G_in, rows, d, w, rstd, G_out, gain, ghat, DTYPE_CODE[dtype])
                                torch.cuda.synchronize()
                                what = (f"{'vit_ln_bwd_full' if full else 'vit_ln_bwd'} d={d} {dtype} x_planes={xp} g={gk} G_in={use_in} "
                                        f"G_out={want_out} ghat={want_hat} gain={gnk}")
                                if want_out:
                                    r = _ratio((G_out.double() - ref).abs(), e)
                                    assert r <= 1.0, (what, "G_out", r)
                                    worst["G_out"] = max(worst["G_out"], r)
                                if want_hat:
                                    gv = gain.double() if gain is not None else 1.0
                                    h64 = ref * gv
                                    eh = e * (gain.double() if gain is not None else 1.0)
                                    if gain is not None:
                                        eh = eh + U * (h64.abs() + eh)
                                    r = _ratio((ghat.double() - h64).abs(), store_bound(h64, eh, dtype, 1))
                                    assert r <= 1.0, (what, "ghat", r)
                                    worst["ghat"] = max(worst["ghat"], r)
                                n += 1
        print(f"REPORT {'vit_ln_bwd_full' if full else 'vit_ln_bwd'} d={d} rows={rows} ({tag}; {n} argument sets): max err/bound "
              f"G_out {worst['G_out']:.3f} ghat {worst['ghat']:.3f}")
        assert n > 0


# =====================================================================================================================
# GELU / QuickGELU
# =====================================================================================================================
def _gelu_inputs(rows, d, pl, dtype, gen):
    """values from -10 to 4 (1 + erf(u / sqrt 2) cancels at the low end), split into planes"""
    v = (torch.rand(rows, d, device="cuda", generator=gen) * 14 - 10).double()
    v[:, :8] = torch.randn(rows, 8, device="cuda", generator=gen).double() * 1e-3
    parts, r = [], v
    for _ in range(pl):
        q = r.to(DT[dtype])
        parts.append(q)
        r = r - q.double()
    return torch.cat(parts, -1)


def _gelu_reference(x, pl, quick):
    """(a, e_a, multiplier, e_mult) in fp64 with absolute bounds (the gate's bound is absolute: 1 + erf cancels near -10)"""
    ef = (pl - 1) * U * x.abs()
    if not quick:
        t = x / math.sqrt(2)
        gate = 0.5 * (1 + torch.special.erf(t))
        dt = t.abs() * (ef / x.abs().clamp_min(1e-300) + 2 * U)             # fl(f * fl(1/sqrt 2))
        egate = 0.5 * (4 * U * torch.special.erf(t).abs() + 2 / math.sqrt(math.pi) * torch.exp(-(t.abs() - dt).clamp_min(0) ** 2) * dt
                       + U * (2 + 4 * U))
        a = x * gate
        ea = x.abs() * egate + gate * ef + U * (a.abs() + x.abs() * egate)
        return a, ea, gate, egate
    k = _f32(1.702)
    z = -k * x
    ez = z.abs() * (ef / x.abs().clamp_min(1e-300) + U)
    ex = torch.exp(z)
    rex = (torch.exp(ez) - 1) + 4 * U * torch.exp(ez)                    # relative error of expf(fl(-k f))
    sg = 1 / (1 + ex)
    rsg = ex / (1 + ex) * rex + 2 * U + 2 * U * rex
    esg = rsg * sg
    a = x * sg
    ea = x.abs() * esg + sg * ef + U * (a.abs() + x.abs() * esg)
    om = 1 - sg
    t = k * x * sg * om
    et = k * (ef * sg * om + x.abs() * (esg * om + sg * (esg + U * om) + esg * (esg + U * om))) + 3 * U * (t.abs() + k * x.abs()
                                                                                                         * (esg + sg) * (om + esg + U))
    dv = sg + t
    edv = esg + et + U * (dv.abs() + esg + et)
    return a, ea, dv, edv


@pytest.mark.gpu
@pytest.mark.parametrize("quick", [False, True], ids=["gelu", "quickgelu"])
@pytest.mark.parametrize("d", [512, 1024, 3072, 200])
def test_vit_gelu_fwd_within_fp64_bound(bcosk_lib, quick, d):
    """vit_gelu_fwd (a = u Phi(u), gain *= Phi(u)) and vit_quickgelu_fwd (a = u sigmoid(1.702 u), gain *= its derivative) over the
    six formats with sq and the gain updated in place (absent / 16-bit / fp32), inputs from -10 to 4 and near 0: a, sq and the gain
    within their bounds (absolute on the gate)."""
    L = _lib()
    rows = 256
    worst = []
    for dtype, pl in FORMATS:
        for gk in (None, "16", "f32"):
            gen = _gen(f"gelu{quick}{d}{dtype}{pl}{gk}")
            u = _gelu_inputs(rows, d, pl, dtype, gen)
            a = torch.full((rows, pl * d), float("nan"), dtype=DT[dtype], device="cuda")
            sq = torch.full((rows,), float("nan"), device="cuda")
            gain = None
            if gk is not None:
                g32 = torch.rand(rows, d, device="cuda", generator=gen) * 2 + 0.01
                gain = g32 if gk == "f32" else g32.to(DT[dtype])
            g_in = None if gain is None else gain.clone()
            (L.vit_quickgelu_fwd if quick else L.vit_gelu_fwd)(u, rows, d, pl, a, sq, gain, DTYPE_CODE[dtype])
            torch.cuda.synchronize()
            what = f"{'vit_quickgelu_fwd' if quick else 'vit_gelu_fwd'} d={d} {dtype}x{pl} gain={gk}"
            x = joined(u, pl, d)
            ref, ea, mult, em = _gelu_reference(x, pl, quick)
            check_residual_planes(a, pl, d, what)
            got = joined(a, pl, d)
            ra = _ratio((got - ref).abs(), store_bound(ref, ea, dtype, pl))
            sq64 = (got * got).sum(-1)
            rs = _ratio((sq.double() - sq64).abs(), (8 * -(-(d // 8) // 32) + 5 + 2 * (pl - 1)) * U * sq64)
            rg = 0.0
            if gain is not None:
                gref = g_in.double() * mult
                eg = g_in.double() * em + U * (gref.abs() + g_in.double() * em)
                b = eg if gk == "f32" else store_bound(gref, eg, dtype, 1)
                rg = _ratio((gain.double() - gref).abs(), b)
            worst.append(f"{dtype}x{pl}/{gk} {ra:.3f}/{rs:.3f}/{rg:.3f}")
            assert ra <= 1.0 and rs <= 1.0 and rg <= 1.0, (what, ra, rs, rg)
    print(f"REPORT {'vit_quickgelu_fwd' if quick else 'vit_gelu_fwd'} d={d} rows={rows}: a / sq / gain max err/bound " + " ".join(worst))


# =====================================================================================================================
# CLIP RN attention-pool head
# =====================================================================================================================
def _sgemm_run(ta, tb, m, n, k, lda, sa, ldb, sb, ldc, sc, batch, alpha, what):
    L = _lib()
    gen = _gen(what)
    ra, ca = (k, m) if ta else (m, k)
    rb, cb = (n, k) if tb else (k, n)
    A = torch.randn((batch - 1) * sa + (ra - 1) * lda + ca, device="cuda", generator=gen)
    B = torch.randn((batch - 1) * sb + (rb - 1) * ldb + cb, device="cuda", generator=gen)
    C = torch.full(((batch - 1) * sc + (m - 1) * ldc + n,), float("nan"), device="cuda")
    L.sgemm_batched(ta, tb, m, n, k, A.data_ptr(), lda, sa, B.data_ptr(), ldb, sb, C.data_ptr(), ldc, sc, batch, alpha)
    torch.cuda.synchronize()
    Am = A.double().as_strided((batch, ra, ca), (sa, lda, 1))
    Bm = B.double().as_strided((batch, rb, cb), (sb, ldb, 1))
    Am = Am.transpose(1, 2) if ta else Am
    Bm = Bm.transpose(1, 2) if tb else Bm
    al = _f32(alpha)
    ref = al * (Am @ Bm)
    T = abs(al) * (Am.abs() @ Bm.abs())
    got = C.double().as_strided((batch, m, n), (sc, ldc, 1))
    r = _ratio((got - ref).abs(), k * U * T + U * ref.abs())
    inside = torch.zeros(C.numel(), dtype=torch.bool, device="cuda")
    inside.as_strided((batch, m, n), (sc, ldc, 1)).fill_(True)
    assert torch.isnan(C[~inside]).all(), (what, "wrote outside C")
    return r


@pytest.mark.gpu
def test_sgemm_batched_within_fp64_bound(bcosk_lib):
    """sgemm_batched at the fused CLIP RN head's own launches and at every (trans_a, trans_b) with both tile widths, ragged m / n / k,
    padded ld and batch strides, alpha != 1: k u sum |a b| |alpha| + u (fma chain, zero-filled tails add exactly)."""
    worst = 0.0
    for key, tag in sorted(_sgemm_plan_geometries().items(), key=str):
        ta, tb, m, n, k, lda, sa, ldb, sb, ldc, sc, batch, alpha = key
        batch = max(batch, 3) if sa and sb and sc else batch
        r = _sgemm_run(ta, tb, m, n, k, lda, sa, ldb, sb, ldc, sc, batch, alpha, f"sgemm plan {key}")
        _report(f"sgemm_batched plan {tag} ta={ta} tb={tb} {m}x{n}x{k} batch={batch} tile={sgemm_tile_width(m, n, batch)}", r)
    for ta, tb, m, n, k, batch, alpha, pad in _sgemm_extra():
        lda = (m if ta else k) + pad
        ldb = (k if tb else n) + pad
        ldc = n + pad
        sa, sb, sc = lda * (k if ta else m) + 7 * pad, ldb * (n if tb else k) + 3 * pad, ldc * m + pad
        r = _sgemm_run(ta, tb, m, n, k, lda, sa, ldb, sb, ldc, sc, batch, alpha, f"sgemm {ta}{tb}{m}{n}{k}{batch}")
        worst = max(worst, r)
        assert r <= 1.0, (ta, tb, m, n, k, batch, r)
    _report(f"sgemm_batched {len(_sgemm_extra())} explicit launches (four transposes x tile 32 / 64, ragged edges)", worst)


@pytest.mark.gpu
def test_head_tokens_and_row_softmax_within_fp64_bound(bcosk_lib):
    """head_tokens at the plan's (npix, c) in the six formats: token j + 1 = the fp32 sum of the planes, token 0 = their mean
    ((planes - 1 + npix - 1) u + u).  row_softmax at the plan's rows and at n = 1, 2, 50, 77, 1000 with one dominant entry per row:
    relative bound (u |s - max| + 4 u of the exponent, the sum's chain, 1 / sum and the product)."""
    L = _lib()
    geoms = {(op.x.shape[1] * op.x.shape[2], op.c) for _, op in opsutil.ops_of(O.HeadTokensOp)}
    assert geoms
    nb = 4
    for npix, c in sorted(geoms):
        worst = []
        for dtype, pl in FORMATS:
            x = _planes_tensor((nb, npix), c, pl, dtype, _gen(f"tok{npix}{c}{dtype}{pl}"))
            tok = torch.full((nb, npix + 1, c), float("nan"), device="cuda")
            L.head_tokens(x, nb, npix, c, pl, DTYPE_CODE[dtype], tok)
            torch.cuda.synchronize()
            xj = joined(x, pl, c)
            r1 = _ratio((tok[:, 1:].double() - xj).abs(), (pl - 1) * U * xj.abs())
            m = xj.mean(1)
            e0 = ((pl - 1) + (npix - 1)) * U * xj.abs().mean(1) + U * m.abs()
            r0 = _ratio((tok[:, 0].double() - m).abs(), e0)
            worst.append(f"{dtype}x{pl} {r1:.3f}/{r0:.3f}")
            assert r1 <= 1.0 and r0 <= 1.0, (npix, c, dtype, pl, r1, r0)
        print(f"REPORT head_tokens npix={npix} c={c} nb={nb}: pixel / mean token max err/bound " + " ".join(worst))
    shapes = {(op.s.numel() // op.s.shape[-1], op.s.shape[-1]) for _, op in opsutil.ops_of(O.RowSoftmaxOp)}
    assert shapes
    for rows, n in sorted(shapes | {(37, 1), (64, 2), (300, 50), (65, 77), (40, 1000)}):
        gen = _gen(f"softmax{rows}{n}")
        s = torch.randn(rows, n, device="cuda", generator=gen) * 4
        dom = torch.randint(0, n, (rows,), device="cuda", generator=gen)
        s[torch.arange(rows, device="cuda")[::2], dom[::2]] += 60.0            # one dominant entry in every other row
        s0 = s.double().clone()
        L.row_softmax(s, rows, n)
        torch.cuda.synchronize()
        ref = torch.softmax(s0, -1)
        z = (s0 - s0.max(-1, keepdim=True).values).abs()
        re = U * z + 4 * U
        chain = -(-n // 32) - 1 + 5
        rel = re + re.max(-1, keepdim=True).values + chain * U + 2 * U
        _report(f"row_softmax rows={rows} n={n}", _ratio((s.double() - ref).abs(), rel * ref))
        if n == 1:
            assert torch.equal(s, torch.ones_like(s)), "a row of one entry must be exactly 1"
