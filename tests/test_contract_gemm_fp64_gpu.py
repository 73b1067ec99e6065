"""-m gpu: the contract-mode GEMM launches against an fp64 evaluation of the same operation, element by element.

The parity mode (the default of every plan) runs on two kernels: the plane-aware kernel (csrc/bcosk_igemm_hp.cu, fp16 x 2
forward and, in `parity_full`, the explanation pass) and the throughput kernel on one fp16 plane (the explanation pass of
`parity`).  tests/test_kernels_gpu.py compares them with tests/emulator.py, which is fp32 and tolerates a maximum over the
tensor; that reference rounds about as much as the error under test.  Here the reference is fp64 and every element has its
own bound, derived from the error model of include/bcosk.h (`hp_accum`).  With u = 2^-24:

Accumulation.  D64 = A @ B^T in fp64 over the launch's own segments (A = the im2col gather, exact 16-bit values), S = |A| @ |B|^T
the sum of |terms| per element.  The tensor core truncates when it aligns an addend to a running sum, so one TMEM accumulation
of L products costs up to L 2^-26 of its sum of |terms|; fp32 round-to-nearest sums of p partials cost p u.
  * plane-aware kernel: the leading segment (a0 b0, sum of |terms| S0) in partials of L = 64 chunk products, the cross terms
    (S - S0 <= 2^-10 S with fp16 planes) in at most one accumulation over their Kx products:
        |D - D64| <= (L 2^-26 + ceil(K0 / L) u) S0 + (Kx 2^-26 + u) (S - S0) + u S
    At K0 = 4608 and chunk 2: 1.9e-6 + 2.1e-6 = 4.0e-6 of S0.
  * throughput kernel: one accumulation over all of K:  |D - D64| <= (K 2^-26 + u) S.
  * bias: the truncation is one-sided, round-to-nearest sums of partials are not, so the bias of the whole sum is that of one
    partial: a one-sided error spread over [0, L 2^-26] has mean L 2^-27, which bounds |mean((D - D64) / S)|.  Measured on positive
    operands (the worst case: every truncation has the same sign) it is 0.26 / 0.32 of L 2^-26 at chunk 2 / 4 (K = 4608); signed
    operands give ~1e-10.  A tighter bound (tau / 16) is not reachable by design: it would require accumulating fewer than 64 products
    per TMEM accumulation, below one K stage.
Epilogue.  The fp64 epilogue of include/bcosk.h runs on D64; the D bound is carried through it by the derivative of every step
(B = 2: y = D |D| inv alpha moves by 2 |D| inv |alpha| per unit of D) plus a few u of the epilogue's own fp32 operations.
Stored outputs add their storage rounding: 2^-11 per fp16 plane (2^-22 for two), 2^-8 / 2^-16 / 2^-24 for one / two / three bf16
planes, u for fp32, and an absolute floor of half the fp16 subnormal spacing (2^-25) per plane.  ReLU / mask bits and MaxOut
indices must match the fp64 decision wherever the fp64 value is farther from the decision point than its own bound.
Plane split.  Every 16-bit plane after the first is the round-to-nearest residual of the planes before it: |p_(i+1)| <= ulp(p_i) / 2.
Rounding of one-plane outputs.  mean((stored - v64) sign(v64) / ulp(stored)) over >= 1e5 elements is ~0 for round-to-nearest and
~-0.5 for truncation; |mean| <= 0.1 is asserted.

Negative controls (numerical variants of real launches, not faults) show that the bounds are tight enough to matter: the whole
leading segment in one TMEM accumulation, and the same data through a one-plane launch, must both be rejected.
"""
import math
import zlib

import pytest
import torch

import emulator as E
import opsutil as U
from bcos_b200 import _lib as L
from bcos_b200.engine import ops as O
from bcos_b200.engine import pack as P
from bcos_b200.engine.base import Act, PlanBase

U24 = 2.0 ** -24
HP_CHUNK_DEFAULT = 2        # bcosk_set_hp_chunk's initial value (checked in test_hp_chunk_bounds)
MEANS6 = (0.485, 0.456, 0.406, 0.515, 0.544, 0.594)
ISTD6 = tuple(1 / s for s in (0.229, 0.224, 0.225, 0.229, 0.224, 0.225))


def _gen(name):
    """generator seeded from the case name (crc32: str hashes are salted per process)"""
    return torch.Generator().manual_seed(zlib.crc32(name.encode()))


# ---------------------------------------------------------------------------------------------------------------------
# fp64 reference
# ---------------------------------------------------------------------------------------------------------------------
def _store_rel(dtype_code: int, planes: int) -> float:
    """relative rounding of a value stored as `planes` 16-bit planes"""
    return 2.0 ** (-(11 if dtype_code == L.DTYPE_CODE["fp16"] else 8) * planes)


def _store_floor(dtype_code: int, planes: int) -> float:
    return planes * 2.0 ** -25 if dtype_code == L.DTYPE_CODE["fp16"] else 0.0


def _seg_cols(op) -> int:
    return len(op.taps) * op.chunks_per_tap * op.kch


def d_bound_coeffs(op, chunk=None):
    """(c0, cx, c): |D - D64| <= c0 S0 + cx (S - S0) + c S for this launch (see the module docstring)"""
    if not op.hp_accum:
        return 0.0, 0.0, op.ktot * 2.0 ** -26 + U24
    k0 = _seg_cols(op)
    L_ = 64 * (chunk or op.hp_chunk or HP_CHUNK_DEFAULT)
    L_ = min(L_, k0)
    kx = op.ktot - k0
    return L_ * 2.0 ** -26 + math.ceil(k0 / L_) * U24, kx * 2.0 ** -26 + U24, U24


def reference_d(op, chunk=None, d_coeff=None):
    """(D64, S, S0, eD) in fp64, [M, n]: the launch's own sum over segments, its sum of |terms|, that of the leading segment
    and the accumulation bound (d_coeff: |D - D64| <= d_coeff S instead of the kernel's model)"""
    A = E.gather_a(op).double()
    B = op.b.double().cpu()
    D = A @ B.t()
    S = A.abs() @ B.abs().t()
    k0 = _seg_cols(op)
    S0 = A[:, :k0].abs() @ B[:, :k0].abs().t()
    c0, cx, c = d_bound_coeffs(op, chunk) if d_coeff is None else (0.0, 0.0, d_coeff)
    return D, S, S0, c0 * S0 + cx * (S - S0) + c * S


def reference_igemm(op, chunk=None, d_coeff=None) -> dict:
    """fp64 evaluation of one IgemmOp (inputs read from the record, which may hold device results copied back) with a bound per
    element for every output.  Returns {name: (value, bound)} plus decision masks: 'pos' / 'pos_amb' (ReLU), 'amax' / 'amax_amb'."""
    M, n = op.M, op.n
    D, S, S0, eD = reference_d(op, chunk, d_coeff)
    out = {"D": (D, eD), "S": S, "S0": S0}
    if op.mode == L.BCOSK_MODE_FWD:
        assert op.act == 0, "fused activations are a throughput-mode option"
        if op.lin_bias is not None:
            D = D + op.lin_bias.double()
            eD = eD + U24 * D.abs()
        einv = 0.0
        inv = None
        if op.scale_mode != L.BCOSK_SCALE_NONE:
            if op.inv_norm is not None:
                inv = op.inv_norm.double()
            else:
                sh, sw, k, st, pd = op.sq_geom
                nb = op.a.shape[0]
                sq = op.sq_in.double().view(op.sq_in.shape[0], nb, 1, sh, sw).sum(0)
                sp = torch.nn.functional.avg_pool2d(sq, k, stride=st, padding=pd, divisor_override=1)
                inv = (1.0 / ((sp + op.sq_eps[0]).sqrt() + op.sq_eps[1])).reshape(-1)
                einv = (k * k * op.sq_in.shape[0] + 4) * U24           # fp32 sum of the window, sqrt, reciprocal
            inv = inv[:, None]
        if op.max_out > 1:
            G = op.max_out
            Dg, eg = D.view(M, n // G, G), eD.view(M, n // G, G)
            top2 = Dg.topk(2, dim=2).values
            best = top2[..., 0]
            idx = (Dg == best[..., None]).double().argmax(dim=2)
            eb = eg.max(dim=2).values
            out["amax"] = idx
            out["amax_amb"] = (top2[..., 0] - top2[..., 1]) <= 2 * eb
            D, eD, n = best, eb, n // G
        alpha = op.alpha.double() if op.alpha is not None else torch.ones(n, dtype=torch.float64)
        beta = op.beta.double() if op.beta is not None else torch.zeros(n, dtype=torch.float64)
        if op.scale_mode == L.BCOSK_SCALE_B2:
            t = D.abs() * inv * alpha
            et = alpha.abs() * inv * eD + t.abs() * (einv + 3 * U24)
            v = D * t + beta
            ev = t.abs() * eD + D.abs() * et + U24 * v.abs()
        elif op.scale_mode == L.BCOSK_SCALE_POW:
            base = D.abs() * inv + 1e-6
            e = op.b_exp - 1.0
            t = base.pow(e) * alpha
            # __powf (ex2 of a scaled lg2): ~2^-18 relative at these magnitudes
            et = alpha.abs() * e * base.pow(e - 1.0) * inv * eD + t.abs() * (2.0 ** -18 + e * einv)
            v = D * t + beta
            ev = t.abs() * eD + D.abs() * et + U24 * v.abs()
        else:
            t = alpha.expand(M, n).clone()
            et = torch.zeros_like(t)
            v = D * alpha + beta
            ev = alpha.abs() * eD + U24 * (D * alpha).abs()
        if op.res is not None:
            r = U._join(op.res.reshape(M, -1).cpu(), op.res_planes)
            ev = ev + 2 * U24 * (v.abs() + r.abs())
            v = v + r
        pos = v > 0
        out["pos"], out["pos_amb"] = pos, v.abs() <= ev
        if op.relu:
            v = torch.where(pos, v, torch.zeros_like(v))
            t = torch.where(pos, t, torch.zeros_like(t))
        out["v"] = (v, ev)
        out["dvdD"] = {L.BCOSK_SCALE_B2: 2 * t.abs(), L.BCOSK_SCALE_POW: op.b_exp * t.abs()}.get(op.scale_mode, t.abs())
        if op.gain is not None:
            gf32 = op.gain.dtype == torch.float32
            eg = et + t.abs() * (U24 if gf32 else _store_rel(op.dtype, 1)) + (0.0 if gf32 else _store_floor(op.dtype, 1))
            out["gain"] = (t, eg)
        yp = 1 if op.y_f32 else op.y_planes
        ey = ev + v.abs() * (U24 if op.y_f32 else _store_rel(op.dtype, yp)) + (0.0 if op.y_f32 else _store_floor(op.dtype, yp))
        out["y"] = (v, ey)
        if op.sq_out is not None:
            bn = op.resolved_block_n() // max(op.max_out, 1)
            parts = []
            for ti in range(op.sq_out.shape[0]):
                vv, ee = v[:, ti * bn:(ti + 1) * bn], ey[:, ti * bn:(ti + 1) * bn]
                s2 = (vv ** 2).sum(1)
                parts.append((s2, (2 * vv.abs() * ee + ee ** 2).sum(1) + vv.shape[1] * U24 * s2 + 1e-30))
            out["sq_out"] = (torch.stack([p[0] for p in parts]), torch.stack([p[1] for p in parts]))
    else:
        rows = E._out_rows(op)
        side = rows if op.side_mapped else torch.arange(M)
        tot, etot = D, eD
        if op.add is not None:
            nb = op.a.shape[0]
            addv = U._join(op.add.cpu(), op.add_planes)
            s = op.add_stride
            full = torch.zeros(nb, op.op, op.oq, n, dtype=torch.float64)
            ap, aq = op.add.shape[1], op.add.shape[2]
            hh, ww = min(op.op, (ap - 1) * s + 1), min(op.oq, (aq - 1) * s + 1)
            full[:, 0:hh:s, 0:ww:s] = addv[:, :(hh + s - 1) // s, :(ww + s - 1) // s]
            full = full.reshape(M, n)
            tot = tot + full
            etot = etot + 2 * U24 * (D.abs() + full.abs())
        if op.out2 is not None:
            o, eo = tot, etot
            if op.mul2 is not None:
                m2 = op.mul2.double().view(-1, n)[side]
                o, eo = o * m2, eo * m2.abs() + U24 * (o * m2).abs()
            if op.mask2 is not None:
                mk = E._mask_bits(op.mask2.cpu(), n)[side]
                o, eo = o * mk, eo * mk
            eo = eo + o.abs() * _store_rel(op.dtype, op.out2_planes) + _store_floor(op.dtype, op.out2_planes)
            out["out2"] = (o, eo)
        v, ev = tot, etot
        if op.mul1 is not None:
            assert op.mul1_sqrt_scale is None
            m1 = op.mul1.double().view(-1, n)[side]
            v, ev = tot * m1, etot * m1.abs() + U24 * (tot * m1).abs()
        out["v"] = (v, ev)
        out["dvdD"] = m1.abs() if op.mul1 is not None else torch.ones_like(v)
        yp = 1 if op.y_f32 else op.y_planes
        out["y"] = (v, ev + v.abs() * (U24 if op.y_f32 else _store_rel(op.dtype, yp))
                    + (0.0 if op.y_f32 else _store_floor(op.dtype, yp)))
    return out


def stored_outputs(op) -> dict:
    """the launch's outputs (record holding device results) as fp64 [M, n] in launch-row order"""
    M = op.M
    rows = E._out_rows(op)
    res = {}
    planes = 1 if op.y_f32 else op.y_planes
    y2 = op.y.reshape(-1, op.y.shape[-1]).cpu()
    assert op.y_col == 0 and y2.shape[-1] % planes == 0
    res["y_planes"] = y2[rows]
    res["y"] = U._join(y2[rows], planes)
    if op.mode == L.BCOSK_MODE_FWD:
        if op.gain is not None:
            res["gain"] = op.gain.cpu().double().view(M, -1)
        if op.maskbits is not None:
            res["mask"] = E._mask_bits(op.maskbits.cpu(), op.n // max(op.max_out, 1))
        if op.amax is not None:
            res["amax"] = op.amax.cpu().long().view(M, -1)
        if op.sq_out is not None:
            res["sq_out"] = op.sq_out.cpu().double()
    elif op.out2 is not None:
        side = rows if op.side_mapped else torch.arange(M)
        o2 = op.out2.reshape(-1, op.out2.shape[-1]).cpu()[side]
        res["out2_planes"] = o2
        res["out2"] = U._join(o2, op.out2_planes)
    return res


def ulp16(x: torch.Tensor, dtype_code: int) -> torch.Tensor:
    """spacing of the 16-bit format above |x| (x representable in it)"""
    fp16 = dtype_code == L.DTYPE_CODE["fp16"]
    _, e = torch.frexp(x.double().abs())
    return torch.ldexp(torch.ones_like(x, dtype=torch.float64), (e - (11 if fp16 else 8)).clamp_min(-24 if fp16 else -133))


def check_plane_split(planes_t: torch.Tensor, planes: int, dtype_code: int, what: str) -> None:
    """every plane after the first is the round-to-nearest residual of the planes before it"""
    c = planes_t.shape[-1] // planes
    for pl in range(1, planes):
        hi = planes_t[..., (pl - 1) * c: pl * c].double()
        lo = planes_t[..., pl * c:(pl + 1) * c].double()
        lim = torch.where(hi == 0, torch.full_like(hi, _store_floor(dtype_code, 1)), ulp16(hi, dtype_code) / 2)
        bad = lo.abs() > lim
        assert not bad.any(), (what, f"plane {pl}", int(bad.sum()), float((lo.abs() / lim.clamp_min(1e-300))[bad].max()))


def check_bounded(name: str, got: torch.Tensor, ref: torch.Tensor, bound: torch.Tensor, scale=None, valid=None) -> dict:
    """|got - ref| <= bound per element; returns the statistics reported for the case"""
    err = (got.double() - ref).abs()
    if valid is not None:
        err, bound, ref = err[valid], bound[valid], ref[valid]
        scale = None if scale is None else scale[valid]
    ratio = err / bound.clamp_min(1e-300)
    worst = float(ratio.max()) if ratio.numel() else 0.0
    if worst > 1.0:
        i = int(ratio.flatten().argmax())
        raise AssertionError(f"{name}: element {i} off by {float(err.flatten()[i]):.3e}, bound {float(bound.flatten()[i]):.3e} "
                             f"(x{worst:.2f}), value {float(ref.flatten()[i]):.6e}")
    st = {"max_err_over_bound": worst}
    if scale is not None:
        sel = scale > 0
        st["max_err_over_S"] = float((err[sel] / scale[sel]).max()) if sel.any() else 0.0
    return st


def check_launch(dev_cpu, chunk=None, label=None, d_coeff=None) -> dict:
    """every output of one launch (record holding device results on the CPU) against its fp64 bounds"""
    label = label or dev_cpu.name
    ref = reference_igemm(dev_cpu, chunk, d_coeff)
    got = stored_outputs(dev_cpu)
    stats = {}
    S = ref["S"]
    if dev_cpu.mode == L.BCOSK_MODE_FWD and dev_cpu.max_out > 1:
        S = S.view(dev_cpu.M, -1, dev_cpu.max_out).max(2).values
    v, ey = ref["y"]
    st = check_bounded(label + ".y", got["y"], v, ey, S if dev_cpu.mode == L.BCOSK_MODE_FWD and dev_cpu.scale_mode == L.BCOSK_SCALE_NONE
                       and dev_cpu.alpha is None and dev_cpu.res is None else None)
    stats["y"] = st["max_err_over_bound"]
    # the error of y in units of S (through the epilogue's derivative): max, signed mean, and the accumulation bound tau
    gS = ref["dvdD"] * S
    sel = (gS > 0) & (v != 0)
    r = (got["y"] - v)[sel] / gS[sel]
    stats["y_err_over_S_max"] = float(r.abs().max()) if r.numel() else 0.0
    stats["y_err_over_S_mean"] = float(r.mean()) if r.numel() else 0.0
    stats["tau"] = sum(d_bound_coeffs(dev_cpu, chunk))
    if not dev_cpu.y_f32 and dev_cpu.y_planes > 1:
        check_plane_split(got["y_planes"], dev_cpu.y_planes, dev_cpu.dtype, label + ".y")
    if "out2" in got:
        o, eo = ref["out2"]
        stats["out2"] = check_bounded(label + ".out2", got["out2"], o, eo)["max_err_over_bound"]
        if dev_cpu.out2_planes > 1:
            check_plane_split(got["out2_planes"], dev_cpu.out2_planes, dev_cpu.dtype, label + ".out2")
    if "gain" in got:
        t, eg = ref["gain"]
        ok = ~ref["pos_amb"] if dev_cpu.relu else None
        stats["gain"] = check_bounded(label + ".gain", got["gain"], t, eg, valid=ok)["max_err_over_bound"]
    if "mask" in got:
        dec = ~ref["pos_amb"]
        want = ref["pos"] if dev_cpu.relu else torch.ones_like(ref["pos"])
        bad = (got["mask"] != want) & dec
        assert not bad.any(), (label, "mask bits", int(bad.sum()))
    if "amax" in got:
        bad = (got["amax"] != ref["amax"]) & ~ref["amax_amb"]
        assert not bad.any(), (label, "MaxOut index", int(bad.sum()))
    if "sq_out" in got:
        s2, es = ref["sq_out"]
        stats["sq_out"] = check_bounded(label + ".sq_out", got["sq_out"], s2, es)["max_err_over_bound"]
    return stats


def run_ops(ops, memo=None):
    memo = {} if memo is None else memo
    dops = [U.to_device(o, "cuda", memo) for o in ops]
    for o in dops:
        o.run()
    torch.cuda.synchronize()
    return dops


def to_cpu(dop):
    return U.to_device(dop, "cpu", {})


def bias_bound(op, chunk=None) -> float:
    """bound on |mean((D - D64) / S)|: half the truncation of one TMEM accumulation (see the module docstring)"""
    if not op.hp_accum:
        return op.ktot * 2.0 ** -27
    return min(64 * (chunk or op.hp_chunk or HP_CHUNK_DEFAULT), _seg_cols(op)) * 2.0 ** -27


def d_stats(dev_cpu, D, D64, S) -> tuple:
    """(max |D - D64| / S, mean (D - D64) / S) over the elements with S > 0"""
    sel = S > 0
    r = (D.double() - D64)[sel] / S[sel]
    return float(r.abs().max()), float(r.mean())


# ---------------------------------------------------------------------------------------------------------------------
# inputs
# ---------------------------------------------------------------------------------------------------------------------
def _act(g, nb, h, w, c, planes, dt, scale=1.0, positive=False):
    v = torch.randn(nb, h, w, c, generator=g) * scale
    if positive:
        v = v.abs()
    t = torch.zeros(nb, h, w, planes * c, dtype=dt)
    stored = E._split_store(t, v, planes)
    sq = (stored.double() ** 2).sum(-1).reshape(1, -1).float().contiguous()
    return Act(t, c, sq, 1)


def _plan(nb, planes=2, dtype="fp16", explain_planes=1, **kw):
    plan = PlanBase(nb, planes=planes, dtype=dtype, device="cpu", explain=True, explain_planes=explain_planes, **kw)
    plan.flat_3x3 = False
    return plan


def _bn(plan, g, cout):
    plan.sd = {"bn.running_var": torch.rand(cout, generator=g) + 0.5, "bn.weight": torch.rand(cout, generator=g) + 0.5}


# forward launches of the plane-aware kernel: name -> emit(plan, g) -> the checked op; the plan comes from `plan_kw`
def _fwd_conv(nb, h, cin, cout, k, stride, *, relu=True, res=False, bn=False, fold=True, a_planes=None, dt=torch.float16,
              **conv_kw):
    def emit(plan, g):
        pa = plan.planes if a_planes is None else a_planes
        x = _act(g, nb, h, h, cin, pa, dt)
        w = torch.randn(cout, cin, k, k, generator=g) / math.sqrt(cin * k * k)
        if bn:
            _bn(plan, g, cout)
        plan.fold_bn = fold
        oh = (h + 2 * (k // 2) - k) // stride + 1
        r = _act(g, nb, oh, oh, cout, conv_kw.get("res_planes", plan.planes), dt) if res else None
        kw = dict(conv_kw)
        if a_planes is not None:
            kw.update(a_planes=a_planes, hp=True)
        plan._conv_fwd("c", x, w, stride, k // 2, k // 2, bn="bn" if bn else None, relu=relu, res=r, want_mask=relu, **kw)
        return plan.fwd_ops
    return emit


FWD_CASES = {
    # name: (plan kwargs, emitter, expected (block_n, paired kind or None))
    "f_1x1_c64_res": (dict(nb=2), _fwd_conv(2, 8, 64, 64, 1, 1, res=True), 64),
    "f_3x3_c64_odd_stages": (dict(nb=2), _fwd_conv(2, 8, 64, 64, 3, 1), 64),
    "f_wide_3x3_s2_c256_mtail": (dict(nb=2), _fwd_conv(2, 14, 256, 128, 3, 2), 128),
    "f_1x1_c1024_bn_res_gain16": (dict(nb=1), _fwd_conv(1, 10, 1024, 256, 1, 1, res=True, bn=True, fold=False), 64),
    "f_1x1_c1024_bn_res_gain32": (dict(nb=1, explain_planes=2), _fwd_conv(1, 10, 1024, 256, 1, 1, res=True, bn=True, fold=False), 64),
    "f_wide_3x3_c256_res": (dict(nb=1), _fwd_conv(1, 10, 256, 256, 3, 1, res=True), 128),
    "f_wide_3x3_c512_res": (dict(nb=1), _fwd_conv(1, 10, 512, 256, 3, 1, res=True), 128),
    "f_vit_residual_add": (dict(nb=2), _fwd_conv(2, 9, 192, 128, 1, 1, relu=False, res=True, a_planes=1, w_planes=2, y_planes=2,
                                                  res_planes=2), 64),
    "f_bf16x3_6seg": (dict(nb=1, planes=3, dtype="bf16", explain_planes=3), _fwd_conv(1, 10, 64, 128, 3, 1, res=True,
                                                                                          dt=torch.bfloat16), 64),
    "f_bf16x2_kch32_unpaired": (dict(nb=2, planes=2, dtype="bf16", explain_planes=2), _fwd_conv(2, 10, 32, 64, 3, 1, dt=torch.bfloat16,
                                                                                                  kch=32), 64),
    "f_pow2p5_bias_maxout2_f32": (dict(nb=2, b=2.5), _fwd_conv(2, 9, 64, 144, 1, 1, relu=False, y_f32=True, max_out=2,
                                                              lin_bias=torch.linspace(-0.1, 0.1, 144)), 64),
    "f_n72_per_row_planes": (dict(nb=2), _fwd_conv(2, 9, 64, 72, 3, 1), 64),
    "f_fc_n1000_f32": (dict(nb=3), _fwd_conv(3, 7, 512, 1000, 1, 1, relu=False, y_f32=True, want_sq=False), 64),
    "f_partial_tile_m49": (dict(nb=1), _fwd_conv(1, 7, 128, 64, 3, 1, res=True), 64),
}


def _emit_fwd(name):
    pkw, emit, bn = FWD_CASES[name]
    pkw = dict(pkw)
    nb = pkw.pop("nb")
    plan = _plan(nb, **pkw)
    ops = emit(plan, _gen(name))
    op = ops[-1]
    assert op.hp_accum and op.resolved_block_n() == bn, (name, op.resolved_block_n())
    return ops


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(FWD_CASES))
def test_hp_forward_fp64(bcosk_lib, name):
    """forward launches of the plane-aware kernel: y planes, gain, mask, sums of squares within the fp64 bounds"""
    ops = _emit_fwd(name)
    dev = to_cpu(run_ops(ops)[-1])
    print("\nTABLE", name, check_launch(dev))


@pytest.mark.gpu
def test_hp_forward_patch_norm_in_kernel(bcosk_lib):
    """`sq_in` with no `inv_norm`: the 3x3 window sum of the producer's sums of squares, inside the epilogue"""
    ops = _emit_fwd("f_3x3_c64_odd_stages")
    assert ops[-1].inv_norm is None and ops[-1].sq_in is not None
    print(check_launch(to_cpu(run_ops(ops)[-1])))


# ---- the kernel's D, observed through a plain linear launch with fp32 output (the CLIP ViT's parity_full launch form)
def _plain_linear(name, cin, n=64, positive=False, nb=2, hw=6, chunk=0):
    g = _gen(name)
    plan = _plan(nb)
    plan.hp_chunk = chunk
    x = _act(g, nb, hw, hw, cin, 2, torch.float16, positive=positive)
    w = torch.randn(n, cin, 1, 1, generator=g) / math.sqrt(cin)
    if positive:
        w = w.abs()
    plan._conv_fwd(name, x, w, 1, 0, 0, bn=None, relu=False, y_f32=True, want_sq=False, scale_mode=L.BCOSK_SCALE_NONE, want_gain=False)
    op = plan.fwd_ops[-1]
    assert op.hp_accum and op.y_f32 and op.gain is None
    return op


def _d_error(op, chunk=None):
    dev = to_cpu(run_ops([op])[0])
    D64, S, S0, eD = reference_d(dev, chunk)
    D = dev.y.reshape(dev.M, dev.n).double()
    c0 = d_bound_coeffs(dev, chunk)[0]
    mx, mean = d_stats(dev, D, D64, S)
    return D, D64, S, eD, c0, mx, mean


@pytest.mark.gpu
@pytest.mark.parametrize("positive", [False, True], ids=["signed", "positive"])
@pytest.mark.parametrize("cin", [576, 4608])
def test_hp_accumulation_bound_and_bias(bcosk_lib, cin, positive):
    """|D - D64| <= tau S per element and |mean (D - D64) / S| <= 64 chunk 2^-27 at the default chunk"""
    op = _plain_linear(f"acc_{cin}_{positive}", cin, positive=positive)
    D, D64, S, eD, c0, mx, mean = _d_error(op)
    print("\nTABLE D", cin, positive, "max |err|/S", mx, "mean", mean, "tau", c0, "bias bound", bias_bound(op))
    check_bounded("D", D, D64, eD)
    assert abs(mean) <= bias_bound(op), (mean, bias_bound(op))


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [1, 2, 4])
def test_hp_chunk_bounds(bcosk_lib, chunk):
    """hp_chunk in {1, 2, 4}: not bit-identical by design, each within its own tau(chunk)"""
    prev = bcosk_lib.bcosk_set_hp_chunk(0)
    bcosk_lib.bcosk_set_hp_chunk(prev)
    assert prev & 0xffff == HP_CHUNK_DEFAULT
    op = _plain_linear("chunk", 4608, positive=True, chunk=chunk)
    D, D64, S, eD, c0, mx, mean = _d_error(op)
    print("\nTABLE chunk", chunk, "max |err|/S", mx, "mean", mean, "tau", c0, "bias bound", bias_bound(op))
    check_bounded("D", D, D64, eD)
    assert abs(mean) <= bias_bound(op)


@pytest.mark.gpu
def test_negative_control_whole_k_accumulation(bcosk_lib):
    """the leading segment in ONE TMEM accumulation (the error hp_chunk exists to prevent) must break the default chunk's D bound
    and its bias bound: positive operands, K = 4608"""
    stages = 4608 // 64
    op = _plain_linear("whole_k", 4608, positive=True, chunk=stages)
    dev = to_cpu(run_ops([op])[0])
    D64, S, S0, eD_default = reference_d(dev, HP_CHUNK_DEFAULT)
    D = dev.y.reshape(dev.M, dev.n).double()
    c0 = d_bound_coeffs(dev, HP_CHUNK_DEFAULT)[0]
    mx, mean = d_stats(dev, D, D64, S)
    print("\nTABLE whole-K: max |err|/S", mx, "mean", mean, "default tau", c0, "default bias bound", bias_bound(dev, HP_CHUNK_DEFAULT))
    assert ((D - D64).abs() > eD_default).any(), "whole-K accumulation passed the default chunk's D bound"
    assert abs(mean) > bias_bound(dev, HP_CHUNK_DEFAULT), "whole-K accumulation passed the bias bound"
    # and it stays within ITS OWN bound (the error model holds for any chunk)
    check_bounded("D whole-K", D, D64, reference_d(dev, stages)[3])


@pytest.mark.gpu
def test_negative_control_one_plane(bcosk_lib):
    """the same convolution through a one-plane launch must break the two-plane output bound"""
    name = "f_1x1_c64_res"
    two = to_cpu(run_ops(_emit_fwd(name))[-1])
    ref = reference_igemm(two)
    plan = _plan(2)
    g = _gen(name)
    x = _act(g, 2, 8, 8, 64, 2, torch.float16)
    w = torch.randn(64, 64, 1, 1, generator=g) / 8
    r = _act(g, 2, 8, 8, 64, 2, torch.float16)
    # the same values, rounded to one plane: one-plane input, weights, residual and output on the throughput kernel
    x1 = Act(x.t[..., :64].clone(), 64, x.sq, 1)
    plan._conv_fwd("one", x1, w, 1, 0, 0, bn=None, relu=True, res=Act(r.t[..., :64].clone(), 64, None, 1), want_mask=True,
                   a_planes=1, w_planes=1, y_planes=1, res_planes=1, hp=False)
    one = to_cpu(run_ops(plan.fwd_ops)[-1])
    v, ey = ref["y"]
    y1 = U._join(one.y.reshape(one.M, -1), 1)
    assert ((y1 - v).abs() > ey).any(), "a one-plane launch passed the two-plane bound"


# ---- the uint8 stem through the exact byte patch matrix (one-plane A x two-plane folded W, paired = 2)
@pytest.mark.gpu
def test_hp_stem_im2col_against_fp64_conv(bcosk_lib):
    """bcosk_stem_im2col_u8 + the folded-weight launch == the fp64 7x7/2 conv of the normalised [x, 1-x] image with the unfolded
    weights (folded-weight algebra, the "1" column at the image border).  The bound adds 2^-22 + u of the weights (fold in fp64,
    fp32 rounding, two fp16 planes) and the subnormal floor of the second weight plane."""
    g = _gen("stem")
    nb, S_, k, st, pd, o = 2, 32, 7, 2, 3, 64
    xu8 = torch.randint(0, 256, (nb, 3, S_, S_), generator=g, dtype=torch.uint8)
    w = torch.randn(o, 6, k, k, generator=g) / math.sqrt(6 * k * k)
    plan = _plan(nb)
    plan._stem_fwd_im2col("stem", xu8, w, w, k, st, pd, bn=None, mean6=MEANS6, inv_std6=ISTD6, s2d_pad=(2, 1), stem_cp=32, want_sq=True)
    gemm = plan.fwd_ops[-1]
    assert gemm.seg_a_choff == [0, 0] and gemm.seg_b_plane == [0, 1]
    dops = run_ops(plan.fwd_ops)
    dev = to_cpu(dops[-1])
    # fp64 conv of the normalised image, unfolded weights
    v = xu8.double() / 255.0
    x6 = torch.cat([v, 1.0 - v], 1)
    xn = (x6 - torch.tensor(MEANS6, dtype=torch.float64).view(1, 6, 1, 1)) * torch.tensor(ISTD6, dtype=torch.float64).view(1, 6, 1, 1)
    D64 = torch.nn.functional.conv2d(xn, w.double(), stride=st, padding=pd).permute(0, 2, 3, 1).reshape(-1, o)
    A = dev.a.reshape(dev.M, -1).double()                          # exact bytes * 2^-6 and the indicators, as the device wrote them
    wf = P.stem_im2col_weight(w, MEANS6, ISTD6, 2.0 ** -6, A.shape[1]).double()
    S = A.abs() @ wf.abs().t()
    c0, cx, c = d_bound_coeffs(dev)
    eD = (c0 + 2.0 ** -22 + U24) * S + (A.abs().sum(1, keepdim=True) * 2.0 ** -25) + c * S
    inv = dops[0].inv_norm.cpu().double()[:, None]                 # the launch's 1/||patch|| (checked against fp64 below)
    t = D64.abs() * inv
    y64 = torch.where(D64 > 0, D64 * t, torch.zeros_like(t))
    ey = 2 * t * eD + 4 * U24 * y64.abs() + y64.abs() * _store_rel(dev.dtype, 2) + _store_floor(dev.dtype, 2)
    got = U._join(dev.y.reshape(dev.M, -1), 2)
    print("\nTABLE stem", check_bounded("stem.y", got, y64, ey))
    check_plane_split(dev.y.reshape(dev.M, -1), 2, dev.dtype, "stem.y")
    sq = torch.nn.functional.avg_pool2d((xn ** 2).sum(1, keepdim=True), k, stride=st, padding=pd, divisor_override=1).reshape(-1)
    inv64 = 1.0 / (sq + 1e-6).sqrt()
    assert float(((inv[:, 0] - inv64).abs() / inv64).max()) < 2e-6


# ---------------------------------------------------------------------------------------------------------------------
# explanation launches
# ---------------------------------------------------------------------------------------------------------------------
GSCALE = 0.25      # output-gradient magnitudes of the plans after the x 4096 seed: O(0.01 .. 1)


def _explain_ops(name, nb, h, cin, cout, k, stride, *, planes, extras=False, classes=False, flat=False, pad=None):
    """forward record + data-gradient launches of one conv; parity plans: planes = 2 (parity_full) or 1 (parity)"""
    g = _gen(name)
    plan = _plan(nb, explain_planes=planes)
    plan.flat_3x3 = flat
    x = _act(g, nb, h, h, cin, 2, torch.float16)
    w = torch.randn(cout, cin, k, k, generator=g) / math.sqrt(cin * k * k)
    p = k // 2 if pad is None else pad
    _, rec = plan._conv_fwd(name, x, w, stride, p, p, bn=None, relu=True, want_mask=True)
    plan._alloc_ghat(rec, classes=classes)
    oh, ow = rec.out_hw
    tmp = torch.zeros(nb, oh, ow, planes * cout, dtype=torch.float16)
    E._split_store(tmp, torch.randn(nb, oh, ow, cout, generator=g) * GSCALE, planes)
    if rec.ghat_map is not None:
        rec.ghat[:, ::stride, ::stride][:, :oh, :ow] = tmp
    else:
        rec.ghat.copy_(tmp)
    dense = stride > 1 and k == 1
    oh2, ow2 = rec.out_hw if dense else rec.in_hw
    M = nb * oh2 * ow2
    yb = torch.zeros(nb, oh2, ow2, planes * cin, dtype=torch.float16)
    mul1 = (torch.rand(M, cin, generator=g) + 0.5).to(plan.gain_dt)
    kw = {}
    if extras:
        kw = dict(add=_act(g, nb, oh2, ow2, cin, planes, torch.float16, scale=GSCALE).t,
                  out2=torch.zeros(nb, oh2, ow2, planes * cin, dtype=torch.float16),
                  mul2=(torch.rand(M, cin, generator=g) + 0.5).to(plan.gain_dt),
                  mask2=torch.randint(-2**31, 2**31 - 1, (M, (cin + 31) // 32), generator=g, dtype=torch.int64).to(torch.int32))
    plan._dgrad(rec, y=yb, mul1=mul1, **kw)
    return plan.bwd_ops


EXPLAIN_HP_CASES = {
    "e_hp_1x1_extras": dict(nb=2, h=8, cin=128, cout=64, k=1, stride=1, extras=True),
    "e_hp_3x3_c64": dict(nb=2, h=8, cin=64, cout=64, k=3, stride=1),
    "e_hp_3x3_s2_classes": dict(nb=2, h=12, cin=64, cout=128, k=3, stride=2, classes=True),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(EXPLAIN_HP_CASES))
def test_hp_explain_fp64(bcosk_lib, name):
    """parity_full explanation launches (fp16 x 2, fp32 producer gain, two-plane extra gradient, out2 / mul2 / mask2; the strided
    3x3 as parity classes with side tensors by mapped row)"""
    ops = _explain_ops(name, planes=2, **EXPLAIN_HP_CASES[name])
    assert all(o.hp_accum for o in ops)
    if EXPLAIN_HP_CASES[name].get("classes"):
        assert len(ops) == 4 and all(o.side_mapped for o in ops)
    memo = {}
    for o in run_ops(ops, memo):
        print("\nTABLE", name, o.name, check_launch(to_cpu(o)))


EXPLAIN_1P_CASES = {
    "e1_1x1": dict(nb=4, h=14, cin=128, cout=256, k=1, stride=1),
    "e1_3x3_flat": dict(nb=8, h=14, cin=64, cout=64, k=3, stride=1, flat=True),
    "e1_3x3_s2_classes": dict(nb=4, h=28, cin=64, cout=128, k=3, stride=2, classes=True),
    "e1_1x1_s2": dict(nb=4, h=28, cin=128, cout=256, k=1, stride=2),
    "e1_extras": dict(nb=4, h=14, cin=128, cout=64, k=1, stride=1, extras=True),
    "e1_long_k_wide": dict(nb=2, h=14, cin=256, cout=512, k=3, stride=1),
}


def _rounding_mean(got, v64, dtype_code):
    """mean((stored - v64) sign(v64) / ulp(stored)) over the non-zero elements: ~0 for round-to-nearest, ~-0.5 for truncation"""
    sel = (v64 != 0) & (got != 0)
    g, v = got[sel].double(), v64[sel]
    return float(((g - v) * v.sign() / ulp16(g, dtype_code)).mean()), int(sel.sum())


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(EXPLAIN_1P_CASES))
def test_fp16_one_plane_explain_fp64(bcosk_lib, name):
    """the `parity` mode's explanation pass: one fp16 plane on the throughput kernel (one TMEM accumulator over K)"""
    cfg = EXPLAIN_1P_CASES[name]
    ops = _explain_ops(name, planes=1, **cfg)
    assert not any(o.hp_accum for o in ops) and all(o.dtype == L.DTYPE_CODE["fp16"] for o in ops)
    if cfg.get("flat"):
        assert ops[-1].flat
    if name == "e1_long_k_wide":
        assert ops[-1].resolved_block_n() == 128 and ops[-1].ktot == 4608
    dops = run_ops(ops)
    tot_n, acc = 0, 0.0
    for o in dops:
        dev = to_cpu(o)
        print("\nTABLE", name, o.name, check_launch(dev))
        ref = reference_igemm(dev)
        got = stored_outputs(dev)
        mean, cnt = _rounding_mean(got["y"], ref["v"][0], dev.dtype)
        acc += mean * cnt
        tot_n += cnt
    assert tot_n >= 1e5, tot_n
    print("\nTABLE", name, "rounding mean / ulp", acc / tot_n, "over", tot_n)
    assert abs(acc / tot_n) <= 0.1


@pytest.mark.gpu
@pytest.mark.parametrize("sched", [1, 2, 3])
def test_fp16_one_plane_explain_schedules(bcosk_lib, sched):
    """the three schedules autotune chooses between (one CTA per tile, persistent strided, persistent row blocks), each against
    fp64 and bit-identical to one another"""
    outs = []
    for s in (1, sched):
        ops = _explain_ops("e1_sched", nb=4, h=14, cin=128, cout=256, k=1, stride=1, planes=1)
        ops[-1].block_n = 64
        ops[-1].sched = s
        dev = to_cpu(run_ops(ops)[-1])
        check_launch(dev)
        outs.append(dev.y.clone())
    assert torch.equal(outs[0], outs[1])


def test_fp64_reference_against_emulator():
    """the fp64 reference and its bound propagation against tests/emulator.py (fp32) on the same records, CPU only: the
    emulator's outputs must lie within the reference's bounds once the accumulation term is widened to fp32's K u"""
    cases = [("f_1x1_c64_res", None), ("f_pow2p5_bias_maxout2_f32", None), ("f_bf16x3_6seg", None), ("f_n72_per_row_planes", None),
             ("f_1x1_c1024_bn_res_gain32", None), ("e_hp_1x1_extras", 2), ("e_hp_3x3_s2_classes", 2), ("e1_extras", 1)]
    for name, eplanes in cases:
        if eplanes is None:
            ops = _emit_fwd(name)
        else:
            cfg = (EXPLAIN_HP_CASES if eplanes == 2 else EXPLAIN_1P_CASES)[name]
            ops = _explain_ops(name, planes=eplanes, **cfg)
        E.run(ops)
        for o in ops:
            if isinstance(o, O.IgemmOp):
                print(name, o.name, check_launch(o, d_coeff=o.ktot * U24))


# ---------------------------------------------------------------------------------------------------------------------
# A/B switches of the plane-aware kernel
# ---------------------------------------------------------------------------------------------------------------------
SWITCH_FWD = ["f_1x1_c64_res", "f_3x3_c64_odd_stages", "f_1x1_c1024_bn_res_gain16", "f_1x1_c1024_bn_res_gain32", "f_vit_residual_add",
              "f_bf16x3_6seg", "f_n72_per_row_planes", "f_fc_n1000_f32"]
SWITCH_EXPLAIN = ["e_hp_1x1_extras", "e_hp_3x3_s2_classes"]
# bcosk_set_hp_boxes settings: bit 0 boxed epilogue I/O, bit 1 generic epilogue, bit 2 no paired stages, bits 8..: 1 + early-input threshold
# (the default: boxes, packed epilogue, paired stages, early inputs up to 4 K stages).  "unpaired" accumulates the cross terms in
# another order (a0 b1 over all of K, then a1 b0, instead of both per stage), so it is held to the fp64 bound, not to identity.
HP_BOX_SETTINGS = {"per_row": 0 | (5 << 8), "generic": 3 | (5 << 8), "early_0": 1 | (1 << 8), "early_all": 1 | (1001 << 8),
                   "unpaired": 5 | (5 << 8)}
HP_BOX_IDENTICAL = ("per_row", "generic", "early_0", "early_all")


def _switch_ops():
    ops = []
    for nm in SWITCH_FWD:
        ops.append((nm, _emit_fwd(nm)))
    for nm in SWITCH_EXPLAIN:
        ops.append((nm, _explain_ops(nm, planes=2, **EXPLAIN_HP_CASES[nm])))
    return ops


def _outputs_of(dev):
    return [t.cpu() for t in (dev.y, dev.gain, dev.maskbits, dev.out2, dev.amax) if t is not None]


@pytest.mark.gpu
def test_hp_boxes_setting_round_trips(bcosk_lib):
    """bcosk_set_hp_boxes returns a value that restores the previous setting when passed back"""
    prev = bcosk_lib.bcosk_set_hp_boxes(3 | (8 << 8))
    try:
        assert bcosk_lib.bcosk_set_hp_boxes(prev) == 3 | (8 << 8)
        assert bcosk_lib.bcosk_set_hp_boxes(prev) == prev
    finally:
        bcosk_lib.bcosk_set_hp_boxes(prev)


@pytest.mark.gpu
def test_hp_switches_bit_identical_and_bounded(bcosk_lib):
    """every bcosk_set_hp_boxes setting and both hp_wide_stages choices: y planes, gains, masks, MaxOut indices bit-identical to
    the default launch, sums of squares within 1e-6 (regrouped), and every variant within the fp64 bounds"""
    def run_all():
        res = {}
        for nm, ops in _switch_ops():
            for o in run_ops(ops):
                dev = to_cpu(o)
                check_launch(dev, label=f"{nm}/{o.name}")
                res[(nm, o.name)] = (_outputs_of(dev), None if dev.sq_out is None else dev.sq_out.clone())
        return res

    base = run_all()
    failures = []
    for label, setting in HP_BOX_SETTINGS.items():
        prev = bcosk_lib.bcosk_set_hp_boxes(setting)
        try:
            outs = run_all()
        finally:
            assert bcosk_lib.bcosk_set_hp_boxes(prev) == setting
        for key, (tens, sq) in outs.items():
            for i, (a, b) in enumerate(zip(tens, base[key][0])):
                if not torch.equal(a, b):
                    failures.append((label, key, i, int((a != b).sum())))
            if sq is not None and label in HP_BOX_IDENTICAL:
                assert U.max_rel_err(sq, base[key][1]) <= 1e-6, (label, key)
    print("differences (setting, launch, output index, elements):", failures)
    assert not [f for f in failures if f[0] in HP_BOX_IDENTICAL], failures


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["f_wide_3x3_c256_res", "f_wide_3x3_c512_res", "f_wide_3x3_s2_c256_mtail"])
def test_hp_wide_stages_bit_identical(bcosk_lib, name):
    """hp_wide_stages 0 (64-wide tiles) and 8 (128-wide tiles) of the same launch: bit-identical y planes and gains"""
    outs = {}
    for wide in (8, 0):
        pkw, emit, _ = FWD_CASES[name]
        pkw = dict(pkw)
        plan = _plan(pkw.pop("nb"), **pkw)
        plan.hp_wide_stages = wide
        op = emit(plan, _gen(name))[-1]
        assert op.resolved_block_n() == (128 if wide else 64)
        dev = to_cpu(run_ops([op])[0])
        check_launch(dev)
        outs[wide] = (_outputs_of(dev), dev.sq_out.sum(0))
    for a, b in zip(outs[8][0], outs[0][0]):
        assert torch.equal(a, b)
    assert U.max_rel_err(outs[8][1], outs[0][1]) < 1e-6
