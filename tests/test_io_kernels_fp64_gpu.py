"""-m gpu: the kernels at the two ends of every plan against an fp64 evaluation of the same operation, element by element.

At the input end: the stem's normalise + space-to-depth (`input_prep_s2d[_u8]`), the patch norms (`patch_inv_norm`) and the ViT
patch rows (`vit_patchify[_u8]`).  At the output end: logits and argmax (`gap_logits`), the explanation seeds (`fc_seed_dgrad`,
`seed_from_nchw`, `seed_from_tokens`), the contribution maps (`contrib_map_s2d[_u8]`, `vit_contrib_map[_u8]`), the RGBA images
(`explanation_rgba[_u8]`) and the localisation scores.  tests/test_kernels_gpu.py compares them with the fp32 emulator at toy sizes
under one flat tolerance; here every reference is fp64, computed from the exact operands the kernel reads (16-bit planes, uint8
pixels, mean / inv_std / scales after rounding to fp32), geometries are collected from the plans, and every element has its own
bound derived from the kernel's order of operations.  With u = 2^-24:

* fp32 roundings: a sum of n non-negative terms (n - 1) u of the sum; a sum of signed terms (n - 1) u of the sum of |terms|;
  products, quotients and sqrt u each; a uint8 pixel x = u8 / 255 and 1 - x are within u of their exact value.
* storage in P 16-bit planes: 2^-11P (fp16) / 2^-8P (bf16) of the value, plus half the fp16 subnormal spacing per plane; every
  later plane is the round-to-nearest residual of the planes before it (|p_(i+1)| <= ulp(p_i) / 2).
* sums of squares (`sq`) are taken over the STORED values (include/bcosk.h): bounded by the fp32 sum alone, far below a storage
  rounding, so a kernel that squared the unrounded values fails.
* explanation_rgba: relative error e_a of the smoothed alpha ((3.5 + 2 (s - 1) + 2) u with an s x s box), order statistics move
  by at most e_a of themselves; the quantile position q (n - 1) is formed in fp32 (q rounded, product rounded: |pos - pos64| <=
  3 u pos64), which moves the interpolated quantile by Q64(pos64 + d) - Q64(pos64 - d), computed from the sorted fp64 alpha.
* decisions (argmax, contribution sign of the alpha channel) must match the fp64 decision wherever the fp64 value is farther from
  the decision point than its bound; inputs are made unambiguous where the test cannot tell.

Every case prints its largest error as a fraction of its bound (REPORT lines, `pytest -s`).
"""
import functools
import math
import zlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import opsutil
from bcos_b200 import _lib as L
from bcos_b200.engine import ops as O

U = 2.0 ** -24
DT = {"fp16": torch.float16, "bf16": torch.bfloat16}
FORMATS = [(dt, pl) for dt in ("fp16", "bf16") for pl in (1, 2, 3)]


def _gen(name, device="cuda"):
    """generator seeded from the case name (crc32: str hashes are salted per process)"""
    return torch.Generator(device=device).manual_seed(zlib.crc32(name.encode()))


def _f32(v) -> float:
    return float(np.float32(v))


def _report(what, ratio):
    print(f"REPORT {what}: max err/bound {ratio:.3f}")
    assert ratio <= 1.0, (what, ratio)


def _ratio(err, bound) -> float:
    return float((err / bound.clamp_min(1e-300)).max()) if err.numel() else 0.0


# ---------------------------------------------------------------------------------------------------------------------
# 16-bit planes
# ---------------------------------------------------------------------------------------------------------------------
_store_rel, _store_floor, _planes, _joined = opsutil.store_rel, opsutil.store_floor, opsutil.split_planes, opsutil.joined
_check_residual_planes, _store_bound = opsutil.check_residual_planes, opsutil.store_bound


@functools.lru_cache(maxsize=None)
def _u8_lut():
    """(x, 1 - x) as the kernels form them from a byte: fp32 division by 255, then fp32 1 - x (IEEE, numpy float32)"""
    v = np.arange(256, dtype=np.float32) / np.float32(255)
    return torch.from_numpy(v.copy()), torch.from_numpy((np.float32(1) - v).astype(np.float32))


def _x6_from_u8(u8):
    """fp32 [nb, 6, h, w] with exactly the values the uint8 kernels compute"""
    a, b = (t.to(u8.device) for t in _u8_lut())
    i = u8.long()
    return torch.cat([a[i], b[i]], 1).contiguous()


def _images(nb, h, w, tag):
    """uint8 RGB [nb, 3, h, w] on the device (synthetic images: smooth structure + noise, every byte value reachable)"""
    g = _gen(tag)
    base = torch.rand(nb, 3, (h + 7) // 8, (w + 7) // 8, device="cuda", generator=g)
    img = F.interpolate(base, size=(h, w), mode="bilinear", align_corners=False) * 230
    img = img + torch.rand(nb, 3, h, w, device="cuda", generator=g) * 25
    img[:, :, 0, 0] = 0
    img[:, :, -1, -1] = 255
    return img.clamp(0, 255).round().to(torch.uint8)


def _x_err(u8_input: bool) -> float:
    """absolute error of the [x, 1 - x] value the kernel forms: u for a byte (x <= 1), 0 for fp32 input"""
    return U if u8_input else 0.0


# ---------------------------------------------------------------------------------------------------------------------
# geometries, from the plans
# ---------------------------------------------------------------------------------------------------------------------
_ops_of = opsutil.ops_of


# =====================================================================================================================
# input end
# =====================================================================================================================
def _input_prep_geometries():
    """{(size, cp, padding (lo, hi) or None, mean6, inv_std6): [tags]} of every InputPrepOp"""
    out = {}
    for tag, op in _ops_of(O.InputPrepOp):
        size = op.x.shape[-1]
        pad = None
        if op.out._base is not None:
            lo = op.out.storage_offset() // (op.out.stride(1) + op.out.stride(2))
            pad = (lo, op.out._base.shape[1] - op.out.shape[1] - lo)
        out.setdefault((size, op.cp, pad, tuple(op.mean6), tuple(op.inv_std6)), []).append(tag)
    return out


def _prep_reference(x6, mean, istd, ex):
    """normalised [x, 1-x] in fp64, space-to-depth order [nb, h/2, w/2, 24], and the fp32 computation's bound"""
    m = torch.tensor([_f32(v) for v in mean], dtype=torch.float64, device=x6.device).view(1, 6, 1, 1)
    s = torch.tensor([_f32(v) for v in istd], dtype=torch.float64, device=x6.device).view(1, 6, 1, 1)
    d = x6.double() - m
    v = d * s
    e = s * (ex + U * (d.abs() + ex)) + U * v.abs()      # fl(x - m), then fl(* istd)
    nb, _, h, w = x6.shape

    def s2d(t):
        return t.view(nb, 6, h // 2, 2, w // 2, 2).permute(0, 2, 4, 3, 5, 1).reshape(nb, h // 2, w // 2, 24)
    return s2d(v), s2d(e)


@pytest.mark.gpu
def test_input_prep_every_plan_geometry_within_fp64_bound(bcosk_lib):
    """input_prep_s2d[_u8] at batch 256 (the whole grid.y) for every (size, cp, layout) the plans launch, in the six formats
    (1 / 2 / 3 planes of fp16 / bf16): values within their bound, planes = round-to-nearest residuals, channels 24..cp exactly
    zero, the border of a padded buffer untouched, and sq = the fp32 sum of the STORED values squared."""
    geoms = _input_prep_geometries()
    assert any(k[0] == 448 for k in geoms) and any(k[2] is not None for k in geoms), geoms
    nb = 256
    for (size, cp, pad, mean, istd), tags in sorted(geoms.items(), key=str):
        u8 = _images(nb, size, size, f"prep{size}")
        for src in ("u8", "f32"):
            x = u8 if src == "u8" else _x6_from_u8(u8) * 0.98 + 0.01        # fp32 input: values between the byte levels
            x6 = _x6_from_u8(u8) if src == "u8" else x
            ref, e = _prep_reference(x6, mean, istd, _x_err(src == "u8"))
            worst = {}
            for dtype, planes in FORMATS:
                h2 = size // 2
                if pad is None:
                    buf = torch.full((nb, h2, h2, planes * cp), float("nan"), dtype=DT[dtype], device="cuda")
                    out = buf
                else:
                    lo, hi = pad
                    buf = torch.full((nb, h2 + lo + hi, h2 + lo + hi, planes * cp), float("nan"), dtype=DT[dtype], device="cuda")
                    out = buf[:, lo:lo + h2, lo:lo + h2, :]
                sq = torch.full((nb * size * size,), float("nan"), device="cuda")
                L.input_prep_s2d(x, mean, istd, out, cp, planes, L.DTYPE_CODE[dtype], sq)
                torch.cuda.synchronize()
                what = f"input_prep {src} {size} cp={cp} pad={pad} {dtype}x{planes}"
                if pad is not None:
                    border = torch.ones(buf.shape[:3], dtype=torch.bool, device="cuda")
                    border[:, lo:lo + h2, lo:lo + h2] = False
                    assert torch.isnan(buf[border].float()).all(), (what, "border written")
                ps = _planes(out, planes, cp)
                for p in ps:
                    assert torch.equal(p[..., 24:], torch.zeros_like(p[..., 24:])), (what, "channels 24..cp not zero")
                _check_residual_planes(out[..., :], planes, cp, what)
                got = sum(p[..., :24].double() for p in ps)
                b = _store_bound(ref, e, dtype, planes)
                rv = _ratio((got - ref).abs(), b)
                # sq of the stored values: 6 fp32 fma roundings of their sum
                st = got.view(nb, h2, h2, 2, 2, 6)
                sq64 = (st * st).sum(-1).permute(0, 1, 3, 2, 4).reshape(nb, size, size).reshape(-1)
                rs = _ratio((sq.double() - sq64).abs(), 6 * U * sq64 + 1e-300)
                worst[f"{dtype}x{planes}"] = (rv, rs)
                assert rv <= 1.0 and rs <= 1.0, (what, rv, rs)
            print(f"REPORT input_prep {src} {size}^2 cp={cp} pad={pad} nb={nb} ({', '.join(sorted(set(tags)))}): value / sq max err/bound "
                  + " ".join(f"{k} {a:.3f}/{s:.3f}" for k, (a, s) in worst.items()))


def _patch_norm_geometries():
    out = set()
    for _, op in _ops_of(O.PatchNormOp):
        out.add((op.parts, op.h, op.w, op.k, op.stride, op.pad, op.eps_in, op.eps_out, op.op, op.oq))
    return sorted(out)


@pytest.mark.gpu
def test_patch_inv_norm_every_plan_geometry_within_fp64_bound(bcosk_lib):
    """patch_inv_norm at every PatchNormOp geometry of the plans (the 7x7/2 stem at 224 and 448 among them), plus the stem
    window over an output that is not a multiple of the 16 x 16 tile and a 3-part sum.  Bound: (k^2 + parts) u relative on the
    window sum, then sqrt, the two epsilons and the reciprocal."""
    geoms = _patch_norm_geometries()
    assert any(g[1] == 448 and g[3] == 7 for g in geoms), geoms
    extra = [(1, 200, 200, 7, 2, 3, 1e-6, 0.0, 100, 100), (3, 58, 58, 7, 2, 3, 1e-6, 0.0, 29, 29)]
    for parts, h, w, k, s, pad, ein, eout, op, oq in geoms + [g for g in extra if g not in geoms]:
        nb = 4
        gen = _gen(f"pn{parts}{h}{k}{s}{pad}")
        sq = torch.rand(parts, nb * h * w, device="cuda", generator=gen) * 4
        sq[:, : h * w // 3] = 0                               # a zero region: the eps terms decide there
        inv = torch.full((nb * op * oq,), float("nan"), device="cuda")
        L.patch_inv_norm(sq, parts, nb, h, w, k, k, s, pad, ein, eout, inv, op, oq)
        torch.cuda.synchronize()
        ssum = F.avg_pool2d(sq.double().sum(0).view(nb, 1, h, w), k, stride=s, padding=pad, divisor_override=1)
        ssum = ssum[:, 0, :op, :oq].reshape(-1)
        e_in, e_out = _f32(ein), _f32(eout)
        r = (ssum + e_in).sqrt()
        ref = 1.0 / (r + e_out)
        # relative: the window sum's (k^2 + parts) u carried through sqrt (half), + eps_in, sqrt, + eps_out, reciprocal
        rel = 0.5 * (k * k + parts) * U * ssum / (ssum + e_in).clamp_min(1e-300) + 4 * U
        ratio = _ratio((inv.double() - ref).abs(), rel * ref)
        _report(f"patch_inv_norm parts={parts} {h}x{w} k={k} s={s} pad={pad} eps=({ein:g}, {eout:g}) -> {op}x{oq}", ratio)


def _patchify_geometries():
    out = set()
    for tag, op in _ops_of(O.VitPatchifyOp):
        out.add((op.x.shape[-2], op.x.shape[-1], op.p, tuple(op.mean6), tuple(op.inv_std6)))
    return sorted(out)


@pytest.mark.gpu
def test_vit_patchify_every_plan_geometry_within_fp64_bound(bcosk_lib):
    """vit_patchify[_u8] at every plan geometry (ViT-Ti 224/16 and 256/16, CLIP ViT 224/32), batch 256, six formats: column
    (p1 p + p2) 6 + c, value bounds, residual planes, and sq = sum of the stored values squared (6 fma + the block's tree)."""
    geoms = _patchify_geometries()
    assert {(g[0], g[2]) for g in geoms} >= {(224, 16), (256, 16), (224, 32)}, geoms
    nb = 256
    for h, w, p, mean, istd in geoms:
        u8 = _images(nb, h, w, f"patchify{h}{p}")
        gh, gw, D = h // p, w // p, p * p * 6
        for src in ("u8", "f32"):
            x = u8 if src == "u8" else _x6_from_u8(u8) * 0.98 + 0.01
            x6 = _x6_from_u8(u8) if src == "u8" else x
            m = torch.tensor([_f32(v) for v in mean], dtype=torch.float64, device="cuda").view(1, 6, 1, 1)
            s = torch.tensor([_f32(v) for v in istd], dtype=torch.float64, device="cuda").view(1, 6, 1, 1)
            ex = _x_err(src == "u8")
            d = x6.double() - m
            v, e = d * s, s * (ex + U * (d.abs() + ex)) + U * (d * s).abs()

            def rows(t):
                return t.view(nb, 6, gh, p, gw, p).permute(0, 2, 4, 3, 5, 1).reshape(nb * gh * gw, D)
            ref, e = rows(v), rows(e)
            worst = []
            for dtype, planes in FORMATS:
                out = torch.full((nb * gh * gw, planes * D), float("nan"), dtype=DT[dtype], device="cuda")
                sq = torch.full((nb * gh * gw,), float("nan"), device="cuda")
                L.vit_patchify(x, p, mean, istd, out, planes, L.DTYPE_CODE[dtype], sq)
                torch.cuda.synchronize()
                what = f"vit_patchify {src} {h}x{w}/{p} {dtype}x{planes}"
                _check_residual_planes(out, planes, D, what)
                got = _joined(out, planes, D)
                rv = _ratio((got - ref).abs(), _store_bound(ref, e, dtype, planes))
                sq64 = (got * got).sum(1)
                depth = 6 + int(math.log2(p * p)) + 1
                rs = _ratio((sq.double() - sq64).abs(), depth * U * sq64)
                worst.append(f"{dtype}x{planes} {rv:.3f}/{rs:.3f}")
                assert rv <= 1.0 and rs <= 1.0, (what, rv, rs)
            print(f"REPORT vit_patchify {src} {h}x{w}/{p} nb={nb}: value / sq max err/bound " + " ".join(worst))


# =====================================================================================================================
# output end: logits, argmax, seeds
# =====================================================================================================================
def _gap_reference(fc, nb, npix, ncls, inv_temp, bias):
    f = fc.double().view(nb, npix, ncls)
    it, b = _f32(inv_temp), _f32(bias)
    ref = f.mean(1) * it + b
    mabs = f.abs().mean(1)
    # sequential fp32 sum of npix terms, * 1/npix (itself rounded), * inv_temp, + bias
    bound = ((npix - 1) * U + 3 * U) * mabs * abs(it) + U * (f.mean(1) * it).abs() + U * ref.abs()
    return ref, bound


@pytest.mark.gpu
@pytest.mark.parametrize("npix,ncls", [(49, 1000), (196, 1000), (197, 1000), (49, 1), (197, 1)])
def test_gap_logits_within_fp64_bound_and_argmax(bcosk_lib, npix, ncls):
    """Logits within npix u sum|fc| inv_temp + the scale and bias roundings; pred = torch.argmax of the kernel's own logits (first
    index on exact ties, crafted below) and = the fp64 argmax wherever the top two are farther apart than twice the bound."""
    nb = 64
    gen = _gen(f"gap{npix}{ncls}")
    fc = torch.randn(nb * npix, ncls, device="cuda", generator=gen)
    fcv = fc.view(nb, npix, ncls)
    if ncls > 1:
        # exact ties: images 0..7 get copies of their best column at three later class indices
        for i in range(8):
            j = 10 + 7 * i
            fcv[i, :, j] += 10.0
            for k in (j + 1, ncls - 1, j + 100):
                fcv[i, :, k % ncls] = fcv[i, :, j]
    inv_temp, bias = 1.0 / 0.7, -math.log(999)
    logits = torch.full((nb, ncls), float("nan"), device="cuda")
    pred = torch.full((nb,), -1, dtype=torch.int32, device="cuda")
    L.gap_logits(fc, nb, npix, ncls, inv_temp, bias, logits, pred)
    torch.cuda.synchronize()
    ref, b = _gap_reference(fc, nb, npix, ncls, inv_temp, bias)
    _report(f"gap_logits npix={npix} ncls={ncls}", _ratio((logits.double() - ref).abs(), b))
    assert torch.equal(pred.long(), logits.argmax(1)), "pred is not the first maximum of the logits"
    if ncls > 1:
        for i in range(8):
            assert pred[i].item() == 10 + 7 * i, (i, pred[i].item())
        top2 = ref.topk(2, dim=1)
        clear = (top2.values[:, 0] - top2.values[:, 1]) > 2 * b.max(1).values
        assert clear[8:].float().mean() > 0.5
        assert torch.equal(pred.long()[clear], ref.argmax(1)[clear])


@pytest.mark.gpu
def test_gap_logits_nan_and_minus_inf_rows_follow_torch_argmax(bcosk_lib):
    """A NaN logit is the maximum (torch.argmax), the first of several NaNs wins, a row of -inf gives class 0: `pred` is always a
    class index the seed kernel may read.  gap_logits alone is safe on such input: it reads fc and writes logits and pred."""
    nb, npix, ncls = 5, 49, 1000
    fc = torch.randn(nb * npix, ncls, device="cuda", generator=_gen("gapnan"))
    fcv = fc.view(nb, npix, ncls)
    fcv[0, 3, 517] = float("nan")
    fcv[1, 0, 700] = float("nan")
    fcv[1, 5, 33] = float("nan")
    fcv[2] = -float("inf")
    fcv[3] = float("nan")
    fcv[4, :, 999] = float("inf")
    logits = torch.empty(nb, ncls, device="cuda")
    pred = torch.full((nb,), -1, dtype=torch.int32, device="cuda")
    L.gap_logits(fc, nb, npix, ncls, 1.0, 0.0, logits, pred)
    torch.cuda.synchronize()
    want = logits.cpu().argmax(1)
    assert want.tolist() == [517, 33, 0, 0, 999]
    assert pred.cpu().long().tolist() == want.tolist()


def _side(shape, kind, dtype, gen):
    """a multiplier operand: None, fp32, or one 16-bit plane (positive, like a gain)"""
    if kind is None:
        return None
    t = torch.rand(shape, device="cuda", generator=gen) * 2 + 0.01
    return t if kind == "f32" else t.to(DT[dtype])


def _maskbits(rows, c, gen):
    words = (c + 31) // 32
    return torch.randint(-2 ** 31, 2 ** 31 - 1, (rows, words), dtype=torch.int64, device="cuda", generator=gen).to(torch.int32)


def _mask_dense(mask, c):
    """[rows, words] int32 bit words -> [rows, c] bool, bit (ch % 32) of word ch / 32"""
    m = mask.long() & 0xffffffff
    ch = torch.arange(c, device=mask.device)
    return ((m[:, ch // 32] >> (ch % 32)) & 1).bool()


def _check_seed_out(out, ref, e_rel, dtype, planes, c, what, zero=None):
    _check_residual_planes(out, planes, c, what)
    got = _joined(out, planes, c)
    if zero is not None:
        assert torch.equal(got[zero], torch.zeros_like(got[zero])), (what, "masked channels not zero")
    r = _ratio((got - ref).abs(), _store_bound(ref, e_rel * ref.abs(), dtype, planes))
    assert r <= 1.0, (what, r)
    return r


FLAGS = [(gain, mul1, mask, out2) for gain in ("f32", "16") for mul1 in (None, "f32", "16") for mask in (False, True)
         for out2 in (False, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("c,npix,ncls", [(40, 49, 1000), (2048, 49, 1000), (192, 197, 1000)])
def test_fc_seed_dgrad_flags_within_fp64_bound(bcosk_lib, c, npix, ncls):
    """fc_seed_dgrad over every flag combination (gain fp32 / 16-bit, mul1 fp32 / 16-bit / none, mask2, out2) in the six formats,
    targets 0 and ncls - 1; c = 40 puts a channel group in the second mask word.  Reference: coef = fl(fl(inv_temp seed_scale) /
    npix) as the host forms it, then coef gain W_fc [mul1] in fp64; 2 u (3 u with mul1) + storage; masked channels exactly 0."""
    nb = 4
    inv_temp, seed_scale = 1.0 / 0.7, 4096.0
    coef = float(np.float32(np.float32(inv_temp) * np.float32(seed_scale)) / np.float32(npix))
    target = torch.tensor([0, ncls - 1, ncls // 2, ncls - 1], dtype=torch.int32, device="cuda")
    worst = {}
    for dtype, planes in FORMATS:
        gen = _gen(f"fcseed{c}{npix}{dtype}{planes}")
        rows = nb * npix
        w_fc = torch.randn(ncls, c, device="cuda", generator=gen)
        gain32 = torch.rand(rows, ncls, device="cuda", generator=gen) + 0.05
        mask = _maskbits(rows, c, gen)
        for gk, mk, use_mask, use_out2 in FLAGS:
            gain = gain32 if gk == "f32" else gain32.to(DT[dtype])
            mul1 = _side((rows, c), mk, dtype, gen)
            out1 = torch.full((rows, planes * c), float("nan"), dtype=DT[dtype], device="cuda")
            out2 = torch.full((rows, planes * c), float("nan"), dtype=DT[dtype], device="cuda") if use_out2 else None
            L.fc_seed_dgrad(target, gain, gk == "f32", w_fc, nb, npix, ncls, c, inv_temp, seed_scale, mul1, mk == "f32", out1,
                            mask if use_mask else None, out2, planes, L.DTYPE_CODE[dtype])
            torch.cuda.synchronize()
            img = torch.arange(rows, device="cuda") // npix
            cls = target.long()[img]
            gsel = gain.double()[torch.arange(rows, device="cuda"), cls]
            g64 = coef * gsel[:, None] * w_fc.double()[cls]
            what = f"fc_seed c={c} npix={npix} {dtype}x{planes} gain={gk} mul1={mk} mask={use_mask} out2={use_out2}"
            ref1 = g64 * (mul1.double() if mul1 is not None else 1.0)
            r = [_check_seed_out(out1, ref1, (3 if mul1 is not None else 2) * U, dtype, planes, c, what + " out1")]
            if use_out2:
                md = _mask_dense(mask, c) if use_mask else torch.ones(rows, c, dtype=torch.bool, device="cuda")
                r.append(_check_seed_out(out2, g64 * md, 2 * U, dtype, planes, c, what + " out2", zero=~md))
            worst[f"{dtype}x{planes}"] = max(worst.get(f"{dtype}x{planes}", 0.0), *r)
    print(f"REPORT fc_seed_dgrad c={c} npix={npix} ncls={ncls} ({len(FLAGS)} flag sets): max err/bound "
          + " ".join(f"{k} {v:.3f}" for k, v in worst.items()))


SEED_FLAGS = [(mul1, mask, mul2, out1, out2) for mul1 in (None, "f32", "16") for mask in (False, True) for mul2 in (None, "f32", "16")
              for out1, out2 in ((True, True), (True, False), (False, True))]


def _seed_geometries():
    out = {}
    for tag, op in _ops_of(O.SeedFromTokensOp) + _ops_of(O.SeedFromNchwOp):
        if isinstance(op, O.SeedFromTokensOp):
            _, t, c = op.g_tokens.shape
            out[("tokens", t - 1, c)] = tag
        else:
            _, c, h, w = op.g.shape
            out[("nchw", h * w, c)] = tag
    return out


@pytest.mark.gpu
def test_seed_from_tokens_and_nchw_flags_within_fp64_bound(bcosk_lib):
    """seed_from_tokens / seed_from_nchw (CLIP RN50 head) at the plan's shapes over mul1 x mask2 x mul2 x (out1, out2) in the six
    formats.  tokens: g = (g[pix + 1] + g[0] fl(1/npix)) scale, 4 u of (|g1| + |g0| / npix) |scale|; nchw: g scale, u; mul: u."""
    geoms = _seed_geometries()
    assert {k[0] for k in geoms} == {"tokens", "nchw"}, geoms
    nb, scale = 4, 4096.0
    for (kind, npix, c), tag in sorted(geoms.items()):
        worst = {}
        for dtype, planes in FORMATS:
            gen = _gen(f"seed{kind}{npix}{c}{dtype}{planes}")
            rows = nb * npix
            mask = _maskbits(rows, c, gen)
            if kind == "tokens":
                gt = torch.randn(nb, npix + 1, c, device="cuda", generator=gen)
                g1, g0 = gt[:, 1:].double().reshape(rows, c), gt[:, :1].double().expand(nb, npix, c).reshape(rows, c)
                g64 = (g1 + g0 / npix) * scale
                eg = 4 * U * (g1.abs() + g0.abs() / npix) * scale
                hw = int(math.isqrt(npix))
            else:
                hw = int(math.isqrt(npix))
                g = torch.randn(nb, c, hw, hw, device="cuda", generator=gen)
                g64 = g.double().permute(0, 2, 3, 1).reshape(rows, c) * _f32(scale)
                eg = U * g64.abs()
            for mk1, use_mask, mk2, use1, use2 in SEED_FLAGS:
                mul1, mul2 = _side((rows, c), mk1, dtype, gen), _side((rows, c), mk2, dtype, gen)
                o1 = torch.full((nb, hw, hw, planes * c), float("nan"), dtype=DT[dtype], device="cuda") if use1 else None
                o2 = torch.full((nb, hw, hw, planes * c), float("nan"), dtype=DT[dtype], device="cuda") if use2 else None
                mk = mask if use_mask else None
                if kind == "tokens":
                    L.seed_from_tokens(gt, nb, npix, c, scale, mul1, o1, mk, mul2, o2, planes, L.DTYPE_CODE[dtype])
                else:
                    L.seed_from_nchw(g, scale, mul1, o1, mk, mul2, o2, planes, L.DTYPE_CODE[dtype])
                torch.cuda.synchronize()
                what = f"seed_from_{kind} npix={npix} c={c} {dtype}x{planes} mul1={mk1} mask={use_mask} mul2={mk2} out1={use1} out2={use2}"
                r = []
                for out, mul, masked in ((o1, mul1, False), (o2, mul2, use_mask)):
                    if out is None:
                        continue
                    m64 = mul.double() if mul is not None else 1.0
                    ref = g64 * m64
                    e = (eg * (m64.abs() if mul is not None else 1.0) + (U * ref.abs() if mul is not None else 0.0))
                    md = _mask_dense(mask, c) if masked else None
                    if md is not None:
                        ref, e = ref * md, e * md
                    out = out.view(rows, planes * c)
                    _check_residual_planes(out, planes, c, what)
                    got = _joined(out, planes, c)
                    if md is not None:
                        assert torch.equal(got[~md], torch.zeros_like(got[~md])), (what, "masked channels not zero")
                    r.append(_ratio((got - ref).abs(), _store_bound(ref, e, dtype, planes)))
                    assert r[-1] <= 1.0, (what, r[-1])
                worst[f"{dtype}x{planes}"] = max(worst.get(f"{dtype}x{planes}", 0.0), *r)
        print(f"REPORT seed_from_{kind} npix={npix} c={c} ({tag}, {len(SEED_FLAGS)} flag sets): max err/bound "
              + " ".join(f"{k} {v:.3f}" for k, v in worst.items()))


# =====================================================================================================================
# output end: contribution maps
# =====================================================================================================================
def _contrib_geometries():
    out = {}
    for tag, op in _ops_of(O.ContribMapOp):
        out.setdefault(("s2d", op.x.shape[-1], op.cp, tuple(op.inv_std6), op.out_scale), tag)
    for tag, op in _ops_of(O.VitContribMapOp):
        out.setdefault(("vit", op.x.shape[-1], op.p, tuple(op.inv_std6), op.out_scale), tag)
    return out


@pytest.mark.gpu
def test_contrib_maps_every_plan_geometry_within_fp64_bound(bcosk_lib):
    """contrib_map_s2d[_u8] (224, 448; cp 32 / 64) and vit_contrib_map[_u8] (patch 16 / 32) at batch 256: grad6 = the fp32 product
    the kernel forms, bit for bit, at every pixel and channel (prefilled with NaN); cmap within the bound of its 6-term fma sum
    (8 u of sum |x g k| + the byte rounding of x); the uint8 entry point returns exactly what the fp32 one does on x6 built from it."""
    geoms = _contrib_geometries()
    assert {k[1] for k in geoms if k[0] == "s2d"} >= {224, 448} and {k[2] for k in geoms if k[0] == "vit"} >= {16, 32}, geoms
    nb = 256
    for (kind, size, cp_or_p, istd, out_scale), tag in sorted(geoms.items(), key=str):
        gen = _gen(f"cmap{kind}{size}{cp_or_p}")
        u8 = _images(nb, size, size, f"cmap{size}")
        x6 = _x6_from_u8(u8)
        is32 = torch.tensor([_f32(v) for v in istd], device="cuda")
        os32 = torch.tensor(_f32(out_scale), device="cuda")
        if kind == "s2d":
            cp, h2 = cp_or_p, size // 2
            g = torch.randn(nb, h2, h2, cp, device="cuda", generator=gen)
            # grad6 as the kernel forms it: g * fl(inv_std * out_scale), the 2x2 sub-pixel (dy, dx) at channel (2 dy + dx) 6 + c
            gk = g[..., :24].view(nb, h2, h2, 2, 2, 6) * (is32 * os32)
            want6 = gk.permute(0, 5, 1, 3, 2, 4).reshape(nb, 6, size, size)
            kfac = (is32.double() * float(os32)).view(1, 6, 1, 1)
            g64 = g[..., :24].double().view(nb, h2, h2, 2, 2, 6).permute(0, 5, 1, 3, 2, 4).reshape(nb, 6, size, size)
            n_round = 2                                      # fl(inv_std * out_scale), fl(g * k)
        else:
            p = cp_or_p
            gh = size // p
            g = torch.randn(nb * gh * gh, p * p * 6, device="cuda", generator=gen)
            gk = (g.view(nb, gh, gh, p, p, 6) * is32) * os32          # fl(fl(g * inv_std) * out_scale)
            want6 = gk.permute(0, 5, 1, 3, 2, 4).reshape(nb, 6, size, size)
            kfac = (is32.double() * float(os32)).view(1, 6, 1, 1)
            g64 = g.double().view(nb, gh, gh, p, p, 6).permute(0, 5, 1, 3, 2, 4).reshape(nb, 6, size, size)
            n_round = 2
        gfull = g64 * kfac
        ref = (x6.double() * gfull).sum(1)
        T = (x6.double().abs() * gfull.abs()).sum(1)
        outs = {}
        for src, x in (("u8", u8), ("f32", x6)):
            cmap = torch.full((nb, size, size), float("nan"), device="cuda")
            grad6 = torch.full((nb, 6, size, size), float("nan"), device="cuda")
            if kind == "s2d":
                L.contrib_map_s2d(g, x, nb, size, size, cp, istd, out_scale, cmap, grad6)
            else:
                L.vit_contrib_map(g, x, p, istd, out_scale, cmap, grad6)
            torch.cuda.synchronize()
            outs[src] = (cmap, grad6)
        cmap, grad6 = outs["u8"]
        assert torch.equal(outs["f32"][0], cmap) and torch.equal(outs["f32"][1], grad6), (kind, size, "u8 and fp32 input differ")
        assert torch.equal(grad6, want6), (kind, size, "grad6 differs from the fp32 product")
        ex = U
        b = (6 + n_round) * U * T + ex * gfull.abs().sum(1) * (1 + 8 * U)
        _report(f"{'contrib_map_s2d' if kind == 's2d' else 'vit_contrib_map'} {size}^2 {'cp' if kind == 's2d' else 'p'}={cp_or_p} "
                f"nb={nb} ({tag})", _ratio((cmap.double() - ref).abs(), b))


# =====================================================================================================================
# output end: RGBA images
# =====================================================================================================================
def _interp(sorted64, pos):
    """torch.quantile's linear interpolation at position pos (float tensor [nb]) of rows sorted64 [nb, n]"""
    n = sorted64.shape[1]
    pos = pos.clamp(0, n - 1)
    lo = pos.floor().long().clamp(0, n - 1)
    hi = (lo + 1).clamp(max=n - 1)
    f = pos - lo.double()
    a, b = sorted64.gather(1, lo[:, None])[:, 0], sorted64.gather(1, hi[:, None])[:, 0]
    return a + (b - a) * f


def _rgba_reference(x6, g, smooth, percentile):
    """fp64 gradient_to_image (bcos/common.py:387-436, oracle.gradient_to_image) per image of the batch, with the per-pixel bound
    of the kernel's alpha channel and colour channels.  Returns (rgb64, e_rgb, alpha64, e_alpha, report dict)."""
    nb, _, h, w = g.shape
    x, lm = x6.double(), g.double()
    contribs = (x * lm).sum(1, keepdim=True)
    rgb = lm / (lm.abs().amax(1, keepdim=True) + 1e-12)
    rgb = rgb.clamp(min=0)
    rgb = rgb[:, :3] / (rgb[:, :3] + rgb[:, 3:] + 1e-12)
    alpha = lm.norm(p=2, dim=1, keepdim=True)
    alpha = torch.where(contribs < 0, torch.zeros_like(alpha) + 1e-12, alpha)
    if smooth:
        alpha = F.avg_pool2d(alpha, smooth, stride=1, padding=(smooth - 1) // 2)
    a = alpha.view(nb, -1)
    n = a.shape[1]
    q = torch.quantile(a, percentile / 100, dim=1, keepdim=True)
    out_a = (alpha / q.view(nb, 1, 1, 1)).clamp(0, 1)[:, 0]
    # ---- bound
    s = smooth if smooth > 1 else 0
    e_a = (3.5 + (2 * (s - 1) + 2 if s else 0)) * U
    pos64 = percentile / 100 * (n - 1)
    d = 3 * U * pos64 + U                                    # fp32 q and q (n - 1)
    srt = a.sort(1).values
    posv = torch.full((nb,), pos64, dtype=torch.float64, device=a.device)
    e_pos = _interp(srt, posv + d) - _interp(srt, posv - d)
    hi_i = torch.full((nb, 1), min(n - 1, math.ceil(pos64 + d) + 1), device=a.device)
    top = srt.gather(1, hi_i)[:, 0]
    e_q = e_a * top + e_pos + 3 * U * top
    qv = q[:, 0]
    e_qrel = torch.where(qv > 0, e_q / qv.clamp_min(1e-300), torch.zeros_like(qv))
    r = (alpha[:, 0] / qv.view(nb, 1, 1))
    rel = (e_a + e_qrel.view(nb, 1, 1)) / (1 - e_qrel.view(nb, 1, 1)) + 2 * U
    e_alpha = r.abs() * rel
    e_rgb = 8 * U * rgb
    return rgb.permute(0, 2, 3, 1), e_rgb.permute(0, 2, 3, 1), out_a, e_alpha, {"e_pos/q": float((e_pos / qv.clamp_min(1e-300)).max())}


def _rgba_inputs(nb, h, w, tag, tied=False):
    gen = _gen(tag)
    u8 = _images(nb, h, w, tag)
    g = torch.randn(nb, 6, h, w, device="cuda", generator=gen)
    if tied:
        # large regions of one gradient vector: alpha has long runs of equal bit patterns (the radix select crosses them)
        blk = torch.randn(nb, 6, (h + 15) // 16, (w + 15) // 16, device="cuda", generator=gen)
        g = blk.repeat_interleave(16, 2).repeat_interleave(16, 3)[:, :, :h, :w].contiguous()
        u8 = torch.full_like(u8, 128)
    x6 = _x6_from_u8(u8)
    # contributions within the fp32 sum's reach of 0 would make the alpha decision ambiguous: zero those gradients
    c = (x6.double() * g.double()).sum(1)
    amb = c.abs() <= 8 * U * (x6.double().abs() * g.double().abs()).sum(1)
    g = g * (~amb)[:, None]
    return u8, x6, g.contiguous()


RGBA_CASES = ([(224, 224, s, 99.5, False) for s in (0, 1, 3, 15)] + [(224, 224, 15, p, False) for p in (0.0, 50.0, 100.0)]
              + [(448, 448, 15, 99.5, False), (448, 448, 0, 50.0, False), (24, 20, 31, 99.5, False),
                 (224, 224, 0, 50.0, True), (224, 224, 15, 99.5, True), (224, 224, 3, 0.0, True)])


@pytest.mark.gpu
@pytest.mark.parametrize("h,w,smooth,percentile,tied", RGBA_CASES)
def test_explanation_rgba_within_fp64_bound(bcosk_lib, h, w, smooth, percentile, tied):
    """explanation_rgba[_u8] against the fp64 restatement of gradient_to_image (torch.quantile in fp64): colour within 8 u of
    itself, alpha within its derived bound (see the module docstring; the fp32 quantile position is bounded, not tolerated);
    the uint8 and fp32 entry points agree bit for bit; image 1 is an all-zero gradient: NaN alpha as in the reference."""
    nb = 16 if h * w <= 224 * 224 else 4
    u8, x6, g = _rgba_inputs(nb, h, w, f"rgba{h}{w}{smooth}{percentile}{tied}", tied)
    g[1] = 0
    outs = []
    for x in (u8, x6):
        tmp = torch.full((2 * nb * h * w + nb,), float("nan"), device="cuda")
        out = torch.full((nb, h, w, 4), -1.0, device="cuda")
        L.explanation_rgba(g, x, smooth, percentile, tmp, out)
        torch.cuda.synchronize()
        outs.append(out)
    assert torch.equal(outs[0].nan_to_num(7.0), outs[1].nan_to_num(7.0)), "uint8 and fp32 input differ"
    out = outs[0]
    rgb, e_rgb, a64, e_a, info = _rgba_reference(x6, g, smooth, percentile)
    assert torch.isnan(a64[1]).all() and torch.isnan(out[1, ..., 3]).all(), "zero gradient image: the reference's 0/0 is NaN"
    assert torch.equal(torch.isnan(out[..., 3]), torch.isnan(a64)), "NaN alpha where the reference has none (or the reverse)"
    ok = ~torch.isnan(a64)
    r_rgb = _ratio((out[..., :3].double() - rgb).abs(), e_rgb + 1e-300)
    r_a = _ratio((out[..., 3].double() - a64).abs()[ok], e_a[ok])
    _report(f"explanation_rgba {h}x{w} nb={nb} smooth={smooth} p={percentile} tied={tied} (quantile position term {info['e_pos/q']:.2e} of q) "
            f"colour", r_rgb)
    _report(f"explanation_rgba {h}x{w} nb={nb} smooth={smooth} p={percentile} tied={tied} alpha", r_a)


# =====================================================================================================================
# output end: localisation scores
# =====================================================================================================================
def _box_bound(v, e, smooth):
    """fp64 zero-padded box sums (horizontal, then vertical and * fl(1/smooth^2)) of v [nt, 1, h, w] with bound propagation"""
    r = smooth // 2
    ones_h = torch.ones(1, 1, 1, smooth, dtype=torch.float64, device=v.device)
    ones_v = torch.ones(1, 1, smooth, 1, dtype=torch.float64, device=v.device)
    v1 = F.conv2d(v, ones_h, padding=(0, r))
    e1 = F.conv2d(e, ones_h, padding=(0, r)) + (smooth - 1) * U * F.conv2d(v.abs(), ones_h, padding=(0, r))
    v2 = F.conv2d(v1, ones_v, padding=(r, 0))
    e2 = F.conv2d(e1, ones_v, padding=(r, 0)) + (smooth - 1) * U * F.conv2d(v1.abs(), ones_v, padding=(r, 0))
    sc = 1.0 / (smooth * smooth)
    return v2 * sc, e2 * sc + 2 * U * (v2 * sc).abs()


def _localisation_geometries():
    """(nt, c, grid, cell): the grid-image path - 2 x 2 and 3 x 3 grids of 224^2 images, one target per cell, attributions
    x * dynamic linear weights (6 channels, ResNetPlan.explain_targets) or contribution maps (1 channel)"""
    return [(4, 6, 2, 224), (4, 1, 2, 224), (9, 6, 3, 224)]


@pytest.mark.gpu
@pytest.mark.parametrize("smooth", [0, 15])
@pytest.mark.parametrize("negate", [False, True])
def test_localisation_scores_within_fp64_bound(bcosk_lib, smooth, negate):
    """localisation_scores at the grid-image geometries, both signs, smoothing 0 / 15, against an fp64 restatement (channel sum,
    box, sign, clamp, region means, fractions) with the bound propagated through every step; a target whose total is <= 0 gives
    exactly 0 in every region."""
    for nt, c, grid, cell in _localisation_geometries():
        h = w = grid * cell
        gen = _gen(f"loc{nt}{c}{grid}{smooth}{negate}")
        attr = torch.randn(nt, c, h, w, device="cuda", generator=gen) * torch.rand(nt, 1, h, w, device="cuda", generator=gen)
        attr[1] = attr[1].abs() * (1 if negate else -1)        # no evidence of the counted sign: total 0
        regions = grid * grid
        tmp = torch.full((2 * nt * h * w + nt * regions,), float("nan"), device="cuda")
        out = torch.full((nt, regions), float("nan"), device="cuda")
        L.localisation_scores(attr, smooth, cell, negate, tmp, out)
        torch.cuda.synchronize()
        a = attr.double()
        v = a.sum(1, keepdim=True)
        e = (c - 1) * U * a.abs().sum(1, keepdim=True)
        if smooth > 1:
            v, e = _box_bound(v, e, smooth)
        if negate:
            v = -v
        v = v.clamp(min=0)
        raw = F.avg_pool2d(v, cell, stride=cell).permute(0, 1, 3, 2).reshape(nt, -1)
        e_raw = (F.avg_pool2d(e, cell, stride=cell) + (cell * cell / 256 + 10) * U * F.avg_pool2d(v, cell, stride=cell))
        e_raw = e_raw.permute(0, 1, 3, 2).reshape(nt, -1)
        total = raw.sum(1, keepdim=True)
        e_tot = e_raw.sum(1, keepdim=True) + (regions / 32 + 6) * U * total
        ref = torch.where(total * raw > 0, raw / total, torch.zeros_like(raw))
        frac_b = (e_raw + ref * e_tot) / (total - e_tot).clamp_min(1e-300) + U * ref
        assert torch.equal(out[1], torch.zeros_like(out[1])), "a target without evidence must score exactly 0"
        keep = torch.ones(nt, dtype=torch.bool, device="cuda")
        keep[1] = False
        _report(f"localisation_scores nt={nt} c={c} grid={grid}x{grid} cell={cell} smooth={smooth} negate={negate}",
                _ratio((out.double() - ref).abs()[keep], frac_b[keep]))
