"""-m gpu: every CUDA kernel (called through the C ABI) against its torch restatement (tests/emulator.py),
on seeded inputs.  Tolerances: 16-bit outputs agree to 1 ulp-ish of bf16 (relative 2^-7 of the tensor max is far
too loose, we use 1.6e-2 only for single-plane bf16 tensors whose last bit may round differently because the
GPU accumulates the fp32 dot products in a different order); fp32 outputs to 2e-5.
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

pytestmark = pytest.mark.gpu

BF16_TOL = 1.0e-2
F32_TOL = 3e-5


def _gen(name):
    """generator seeded from the case name; crc32, not hash(): str hashes are salted per process, so each run would draw
    other inputs"""
    return torch.Generator().manual_seed(zlib.crc32(name.encode()))


def _mini_plan(nb, planes, explain=True, b=2.0):
    plan = PlanBase(nb, planes=planes, dtype="bf16", device="cpu", explain=explain, b=b)
    plan.flat_3x3 = False      # the per-kernel tests choose the gather explicitly (flat=True where they want it)
    return plan


def _rand_act(g, nb, h, w, c, planes, dt=torch.bfloat16, scale=1.0):
    v = torch.randn(nb, h, w, c, generator=g) * scale
    t = torch.zeros(nb, h, w, planes * c, dtype=dt)
    stored = E._split_store(t, v, planes)
    sq = (stored ** 2).sum(-1).reshape(1, -1).contiguous()
    return Act(t, c, sq, 1)


def _run_and_compare(ops, tol16=BF16_TOL, tol32=None):
    # fp32 side outputs computed FROM single-plane bf16 data (sums of squares, logits of rounded inputs) inherit the
    # 1-ulp bf16 differences caused by the different fp32 accumulation order on the GPU
    tol32 = tol32 if tol32 is not None else (5e-3 if tol16 >= 1e-3 else F32_TOL)
    memo = {}
    dev_ops = [U.to_device(o, "cuda", memo) for o in ops]
    E.run(ops)
    for o in dev_ops:
        o.run()
    torch.cuda.synchronize()
    out = {}
    for r, d in zip(ops, dev_ops):
        for name in U.OUTPUT_FIELDS[type(r)]:
            t = getattr(r, name)
            if t is None:
                continue
            tol = tol32 if t.dtype == torch.float32 else tol16
            out[(r.name, name)] = U.compare(r, d, tol, [name])[name]
    return out


CONV_CASES = [
    # name, nb, h, cin, cout, k, stride, pad_lo, pad_hi, planes, relu, res, kch
    ("1x1_c64", 2, 16, 64, 64, 1, 1, 0, 0, 1, True, False, 64),
    ("1x1_c128_n256_res", 2, 12, 128, 256, 1, 1, 0, 0, 1, True, True, 64),
    ("3x3_c64", 2, 14, 64, 64, 3, 1, 1, 1, 1, True, False, 64),
    ("3x3_s2_c64_n128", 2, 14, 64, 128, 3, 2, 1, 1, 1, True, False, 64),
    ("3x3_odd_hw", 3, 7, 128, 128, 3, 1, 1, 1, 1, False, False, 64),
    ("1x1_s2", 2, 14, 128, 256, 1, 2, 0, 0, 1, False, False, 64),
    ("4x4_asym_kch32", 2, 20, 32, 64, 4, 1, 2, 1, 1, True, False, 32),
    ("3x3_planes2", 2, 10, 64, 64, 3, 1, 1, 1, 2, True, True, 64),
    ("3x3_planes3", 1, 10, 64, 128, 3, 1, 1, 1, 3, True, False, 64),
    ("1x1_cin96_tail", 2, 9, 96, 72, 1, 1, 0, 0, 1, True, False, 64),
    ("4x4_asym_kch32_planes3", 1, 12, 32, 64, 4, 1, 2, 1, 3, True, False, 32),
]


@pytest.mark.parametrize("case", CONV_CASES, ids=[c[0] for c in CONV_CASES])
def test_igemm_forward(bcosk_lib, case):
    name, nb, h, cin, cout, k, stride, plo, phi, planes, relu, use_res, kch = case
    g = _gen(name)
    plan = _mini_plan(nb, planes)
    x = _rand_act(g, nb, h, h, cin, planes)
    w = torch.randn(cout, cin, k, k, generator=g) / math.sqrt(cin * k * k)
    plan.sd = {"bn.running_var": torch.rand(cout, generator=g) + 0.5, "bn.weight": torch.rand(cout, generator=g) + 0.5}
    oh = (h + plo + phi - k) // stride + 1
    res = _rand_act(g, nb, oh, oh, cout, planes) if use_res else None
    inv_norm = (torch.rand(nb * oh * oh, generator=g) + 0.5) if plo != phi else None   # asymmetric pad: norm given
    y, rec = plan._conv_fwd(name, x, w, stride, plo, phi, bn="bn", relu=relu, res=res, want_mask=True, kch=kch,
                            inv_norm=inv_norm)
    errs = _run_and_compare(plan.fwd_ops, tol16=BF16_TOL if planes == 1 else 2e-4)
    print(name, errs)


def test_igemm_forward_fc_f32_tail(bcosk_lib):
    """classifier-like: n = 1000 (partial last tile), fp32 output, no BN/ReLU"""
    g = torch.Generator().manual_seed(7)
    plan = _mini_plan(3, 1)
    x = _rand_act(g, 3, 7, 7, 256, 1)
    w = torch.randn(1000, 256, 1, 1, generator=g) / 16
    plan._conv_fwd("fc", x, w, 1, 0, 0, bn=None, relu=False, y_f32=True, want_sq=False)
    print(_run_and_compare(plan.fwd_ops))


def test_igemm_forward_general_b(bcosk_lib):
    g = torch.Generator().manual_seed(8)
    plan = _mini_plan(2, 1, b=2.5)
    x = _rand_act(g, 2, 8, 8, 64, 1)
    w = torch.randn(64, 64, 3, 3, generator=g) / 24
    plan._conv_fwd("b2p5", x, w, 1, 1, 1, bn=None, relu=False)
    print(_run_and_compare(plan.fwd_ops, tol32=2e-4))


@pytest.mark.parametrize("planes", [1, 2])
def test_igemm_forward_plain_linear(bcosk_lib, planes):
    """scale mode NONE per launch (the ViT's to_qkv, bcos/models/vit.py:140): y = W x (+ residual), no gain, packed epilogue"""
    g = torch.Generator().manual_seed(21)
    plan = _mini_plan(2, planes)
    x = _rand_act(g, 2, 6, 6, 128, planes)
    w = torch.randn(192, 128, 1, 1, generator=g) / math.sqrt(128)
    res = _rand_act(g, 2, 6, 6, 192, planes)
    for r in (None, res):
        plan.fwd_ops.clear()
        y, rec = plan._conv_fwd("plain", x, w, 1, 0, 0, bn=None, relu=False, res=r, want_sq=False, scale_mode=L.BCOSK_SCALE_NONE,
                                want_gain=False)
        assert rec.gain is None
        print(_run_and_compare(plan.fwd_ops, tol16=BF16_TOL if planes == 1 else 2e-4))


@pytest.mark.parametrize("k,cin,n,res,relu,pa", [(3, 128, 256, False, True, 2), (1, 1024, 256, True, True, 2), (1, 512, 384, True, False, 1),
                                                 (3, 64, 128, False, True, 2)])
def test_igemm_hp_wide_tiles(bcosk_lib, k, cin, n, res, relu, pa):
    """128-wide tiles of the plane-aware kernel (long K loops: 64 KB paired stages, one CTA per SM, two column groups per epilogue
    warp): same numbers as the 64-wide launch of the same convolution, and both against the emulator"""
    g = torch.Generator().manual_seed(61 + k + n)
    outs = {}
    for wide in (8, 0):
        plan = PlanBase(2, planes=2, dtype="fp16", device="cpu", explain=True, explain_planes=1)
        plan.flat_3x3 = False
        plan.hp_wide_stages = wide
        gg = torch.Generator().manual_seed(61 + k + n)
        x = _rand_act(gg, 2, 10, 10, cin, pa, dt=torch.float16)
        w = torch.randn(n, cin, k, k, generator=gg) / math.sqrt(cin * k * k)
        r = _rand_act(gg, 2, 10, 10, n, 2, dt=torch.float16) if res else None
        kw = dict(a_planes=1, w_planes=2, y_planes=2, res_planes=2, hp=True) if pa == 1 else {}
        y, rec = plan._conv_fwd("wide", x, w, 1, k // 2, k // 2, bn=None, relu=relu, res=r, want_sq=True, want_mask=relu, **kw)
        op = plan.fwd_ops[-1]
        assert op.hp_accum and op.resolved_block_n() == (128 if wide else 64), op.resolved_block_n()
        print(_run_and_compare(plan.fwd_ops, tol16=6e-4))           # (the one-plane fp16 gain: 2^-11)
        dev = U.to_device(op, "cuda", {})
        dev.run()
        torch.cuda.synchronize()
        outs[wide] = (dev.y.clone(), dev.gain.clone(), dev.sq_out.sum(0).clone(), None if dev.maskbits is None else dev.maskbits.clone())
    assert torch.equal(outs[8][0], outs[0][0]) and torch.equal(outs[8][1], outs[0][1])          # y planes and gains: bit-identical
    assert outs[8][3] is None or torch.equal(outs[8][3], outs[0][3])
    assert U.max_rel_err(outs[8][2], outs[0][2]) < 1e-6                                         # per-tile partials regroup the same squares


@pytest.mark.parametrize("act", [1, 2])
@pytest.mark.parametrize("dt,n", [("fp16", 384), ("bf16", 128), ("fp16", 64)])
def test_igemm_forward_fused_gelu(bcosk_lib, dt, n, act):
    """include/bcosk.h `act` = 1: MyGELU (bcos/models/vit.py:89-113) behind the B-cos transform of a one-plane linear launch - y is the
    activation, sq_out its per-tile sums of squares, the gain carries the detached gate (the ViT MLP's linear1); `act` = 2: QuickGELU
    of the CLIP ViT MLP (CLIP/clip/model.py:166-168), whose derivative goes into the gain"""
    g = torch.Generator().manual_seed(51)
    tdt = torch.float16 if dt == "fp16" else torch.bfloat16
    plan = PlanBase(2, planes=1, dtype=dt, device="cpu", explain=True)
    x = _rand_act(g, 2, 7, 9, 192, 1, dt=tdt)
    w = torch.randn(n, 192, 1, 1, generator=g) * (3.0 / math.sqrt(192))          # outputs on both sides of the gate's knee
    y, rec = plan._conv_fwd("gelu", x, w, 1, 0, 0, bn=None, relu=False, sq_eps=(0.0, 1e-12), want_sq=True, act=act)
    assert plan.fwd_ops[-1].act == act and rec.gain is not None and y.sq is not None
    print(_run_and_compare(plan.fwd_ops, tol16=BF16_TOL if dt == "bf16" else 2e-3))
    # against the two-step form (transform, then GELU on the fp32 value): same numbers by construction of the emulator; and the
    # library refuses the combinations the packed epilogue does not implement
    bad = plan.fwd_ops[-1]
    dev = U.to_device(bad, "cuda", {})
    dev.relu = True
    with pytest.raises(L.BcoskError):
        dev.run()


@pytest.mark.parametrize("dt", ["fp16", "bf16"])
def test_stem_im2col_u8(bcosk_lib, dt):
    """bcosk_stem_im2col_u8: byte patch matrix (v_R, v_G, v_B, 1 per in-image tap) and 1/||patch|| of the normalised window"""
    g = torch.Generator().manual_seed(31)
    x = torch.randint(0, 256, (2, 3, 40, 40), generator=g, dtype=torch.uint8)
    mean6, istd6 = (0.485, 0.456, 0.406, 0.515, 0.544, 0.594), tuple(1 / s for s in (0.229, 0.224, 0.225, 0.229, 0.224, 0.225))
    tdt = torch.float16 if dt == "fp16" else torch.bfloat16
    for k, st, pd in ((7, 2, 3), (3, 2, 1)):
        op_ = (40 + 2 * pd - k) // st + 1
        kp = (4 * k * k + 63) // 64 * 64
        op = O.StemIm2colOp("im2col", x, k, st, pd, mean6, istd6, 2.0 ** -6, torch.zeros(2, op_, op_, kp, dtype=tdt), torch.zeros(2 * op_ * op_),
                            L.DTYPE_CODE[dt])
        dev = U.to_device(op, "cuda", {})
        E.run([op])
        dev.run()
        torch.cuda.synchronize()
        assert torch.equal(dev.out.cpu(), op.out)                                   # bytes and indicators are exact
        assert U.max_rel_err(dev.inv_norm, op.inv_norm) < 2e-6


@pytest.mark.parametrize("k,res", [(1, True), (3, False), (1, False)])
def test_igemm_forward_mixed_planes(bcosk_lib, k, res):
    """one-plane input x two-plane weights -> two-plane output (+ two-plane residual) through the plane-aware kernel: the launch format of
    the ViT plans' adds into the residual stream (segments a0 b0 + a0 b1; paired stages without the a1 box)"""
    g = torch.Generator().manual_seed(41 + k)
    plan = PlanBase(2, planes=2, dtype="fp16", device="cpu", explain=True)
    plan.flat_3x3 = False
    x = _rand_act(g, 2, 9, 9, 192, 1, dt=torch.float16)
    w = torch.randn(128, 192, k, k, generator=g) / math.sqrt(192 * k * k)
    r = _rand_act(g, 2, 9, 9, 128, 2, dt=torch.float16) if res else None
    plan._conv_fwd("mixed", x, w, 1, k // 2, k // 2, bn=None, relu=False, res=r, want_sq=True, a_planes=1, w_planes=2, y_planes=2,
                   res_planes=2, hp=True)
    op = plan.fwd_ops[-1]
    assert len(op.seg_a_choff) == 2 and op.seg_a_choff == [0, 0] and op.seg_b_plane == [0, 1] and op.y_planes == 2
    print(_run_and_compare(plan.fwd_ops, tol16=2e-5, tol32=2e-5))
    # and the all-one-plane branch format on the throughput kernel
    plan.fwd_ops.clear()
    plan._conv_fwd("branch", x, w, 1, k // 2, k // 2, bn=None, relu=False, want_sq=True, a_planes=1, w_planes=1, y_planes=1, hp=False)
    print(_run_and_compare(plan.fwd_ops, tol16=2e-3, tol32=2e-3))


MAXOUT_CASES = [
    # name, planes, G, cout (GEMM columns), k, b, bias, y_f32
    ("mo2_1plane_16bit", 1, 2, 128, 3, 2.0, False, False),
    ("mo4_1plane_f32_bias", 1, 4, 64, 1, 2.0, True, True),
    ("mo2_hp3_f32", 3, 2, 64, 3, 2.0, False, True),
    ("mo8_hp3_f32_b2p5_bias", 3, 8, 72, 1, 2.5, True, True),
    ("mo2_hp2_planes_out", 2, 2, 128, 1, 2.0, False, False),
]


@pytest.mark.parametrize("case", MAXOUT_CASES, ids=[c[0] for c in MAXOUT_CASES])
def test_igemm_forward_maxout_in_epilogue(bcosk_lib, case):
    """include/bcosk.h `max_out`: adjacent-column maximum + scale of the kept unit + kept index inside the conv launch
    (bcosconv2d.py:166-170), generic epilogue of the throughput kernel and of the parity-mode kernel."""
    name, planes, G, cout, k, b, bias, y_f32 = case
    g = _gen(name)
    plan = _mini_plan(2, planes, b=b)
    x = _rand_act(g, 2, 9, 9, 64, planes)
    w = torch.randn(cout, 64, k, k, generator=g) / math.sqrt(64 * k * k)
    lb = torch.randn(cout, generator=g) * 0.1 if bias else None
    y, rec = plan._conv_fwd(name, x, w, 1, k // 2, k // 2, bn=None, relu=False, y_f32=y_f32, lin_bias=lb, max_out=G)
    assert y.t.shape[-1] == (1 if y_f32 else planes) * cout // G and rec.gain.shape[-1] == cout // G and rec.amax.shape[-1] == cout // G
    errs = _run_and_compare(plan.fwd_ops, tol16=BF16_TOL if planes == 1 else 2e-4, tol32=2e-4 if (planes > 1 or b != 2.0) else None)
    print(name, errs)


DGRAD_CASES = [
    # name, nb, h_in, cin, cout, k, stride, pad, planes
    ("d_1x1", 2, 12, 64, 128, 1, 1, 0, 1),
    ("d_3x3", 2, 12, 64, 64, 3, 1, 1, 1),
    ("d_3x3_s2_zero_insert", 2, 12, 64, 128, 3, 2, 1, 1),
    ("d_1x1_s2", 2, 12, 128, 256, 1, 2, 0, 1),
    ("d_3x3_planes2", 1, 8, 64, 64, 3, 1, 1, 2),
    ("d_4x4_asym_n32_f32", 2, 16, 32, 64, 4, 1, 2, 1),
]


@pytest.mark.parametrize("case", DGRAD_CASES, ids=[c[0] for c in DGRAD_CASES])
def test_igemm_explain_dgrad(bcosk_lib, case):
    name, nb, h, cin, cout, k, stride, pad, planes = case
    g = _gen(name)
    plan = _mini_plan(nb, planes)
    pad_hi = pad if k != 4 else 1
    x = _rand_act(g, nb, h, h, cin, planes)
    w = torch.randn(cout, cin, k, k, generator=g) / math.sqrt(cin * k * k)
    inv_norm = (torch.rand(nb * ((h + pad + pad_hi - k) // stride + 1) ** 2, generator=g) + 0.5) if pad != pad_hi else None
    y, rec = plan._conv_fwd(name, x, w, stride, pad, pad_hi, bn=None, relu=True, want_mask=True, inv_norm=inv_norm,
                            kch=32 if cin == 32 else 64)
    plan._alloc_ghat(rec)
    # fill ghat (dense positions only when zero-inserted)
    oh, ow = rec.out_hw
    gv = torch.randn(nb, oh, ow, cout, generator=g)
    tmp = torch.zeros(nb, oh, ow, planes * cout, dtype=plan.dt)
    E._split_store(tmp, gv, planes)
    if rec.ghat_map is not None:
        rec.ghat[:, ::stride, ::stride][:, :oh, :ow] = tmp
    else:
        rec.ghat.copy_(tmp)
    f32 = name.endswith("f32")
    dense = stride > 1 and k == 1
    oh2, ow2 = (rec.out_hw if dense else rec.in_hw)
    M = nb * oh2 * ow2
    yb = torch.zeros(nb, oh2, ow2, (1 if f32 else planes) * cin, dtype=torch.float32 if f32 else plan.dt)
    mul1 = None if f32 else (torch.rand(M, cin, generator=g) + 0.5).to(plan.gain_dt)
    add = None if f32 else _rand_act(g, nb, oh2, ow2, cin, planes).t
    out2 = None if f32 else torch.zeros(nb, oh2, ow2, planes * cin, dtype=plan.dt)
    mul2 = None if f32 else (torch.rand(M, cin, generator=g) + 0.5).to(plan.gain_dt)
    mask2 = None if f32 else torch.randint(-2**31, 2**31 - 1, (M, (cin + 31) // 32), generator=g, dtype=torch.int64).to(torch.int32)
    plan._dgrad(rec, y=yb, mul1=mul1, add=add, out2=out2, mul2=mul2, mask2=mask2, y_f32=f32)
    errs = _run_and_compare(plan.bwd_ops, tol16=BF16_TOL if planes == 1 else 2e-4)
    print(name, errs)


def _padded_act(plan, g, nb, h, w, c, lo, hi):
    """random activation stored in the interior view of a zero-bordered buffer (flat-window operand layout)"""
    t = plan._padded(nb, h, w, c, lo, hi)
    v = torch.randn(nb, h, w, c, generator=g)
    t.copy_(v.to(t.dtype))
    sq = (t.float() ** 2).sum(-1).reshape(1, -1).contiguous()
    return Act(t, c, sq, 1)


FLAT_FWD_CASES = [
    # name, nb, h, w, cin, cout, k, pad_lo, pad_hi, kch, relu
    ("flat_4x4_stem_like", 3, 20, 20, 32, 64, 4, 2, 1, 32, True),
    ("flat_4x4_wide_rows", 2, 9, 100, 32, 64, 4, 2, 1, 32, True),      # rows almost as long as a tile
    ("flat_3x3_c64", 2, 14, 14, 64, 64, 3, 1, 1, 64, True),
    ("flat_3x3_n32", 2, 11, 13, 64, 32, 3, 1, 1, 64, False),
    ("flat_1x1_c64", 2, 12, 12, 64, 64, 1, 0, 0, 64, True),
    # dense input (a_flat = 2): the zero borders are made in shared memory by the TMA box
    ("flatdense_3x3_c64_w56", 2, 10, 56, 64, 64, 3, 1, 1, 64, True),
    ("flatdense_3x3_c64_w13", 3, 11, 13, 64, 64, 3, 1, 1, 64, True),
    ("flatdense_3x3_n32_w30", 2, 9, 30, 64, 32, 3, 1, 1, 64, False),
    ("flatdense_4x4_kch32", 2, 20, 20, 32, 64, 4, 2, 1, 32, True),
]


@pytest.mark.parametrize("case", FLAT_FWD_CASES, ids=[c[0] for c in FLAT_FWD_CASES])
def test_igemm_flat_window_forward(bcosk_lib, case):
    """flat-window gather (one shared-memory window per tile, shifted descriptors per tap) == the emulator's conv"""
    name, nb, h, wd, cin, cout, k, plo, phi, kch, relu = case
    g = _gen(name)
    plan = _mini_plan(nb, 1)
    x = _rand_act(g, nb, h, wd, cin, 1) if name.startswith("flatdense") else _padded_act(plan, g, nb, h, wd, cin, plo, phi)
    w = torch.randn(cout, cin, k, k, generator=g) / math.sqrt(cin * k * k)
    oh, ow = h + plo + phi - k + 1, wd + plo + phi - k + 1
    inv_norm = torch.rand(nb * oh * ow, generator=g) + 0.5
    plan.sd = {"bn.running_var": torch.rand(cout, generator=g) + 0.5, "bn.weight": torch.rand(cout, generator=g) + 0.5}
    for fold in (True, False):         # BN folded into the weights / applied as alpha in the epilogue
        plan.fold_bn = fold
        plan.fwd_ops.clear()
        plan._conv_fwd(name, x, w, 1, plo, phi, bn="bn", relu=relu, want_mask=True, kch=kch, inv_norm=inv_norm, flat=True)
        assert plan.fwd_ops[-1].flat
        print(name, fold, _run_and_compare(plan.fwd_ops))


@pytest.mark.parametrize("case", [("flat_d_4x4_n32_f32", 2, 18, 32, 64, 4, 2, 1, True),
                                  ("flat_d_3x3_n64", 2, 12, 64, 64, 3, 1, 1, False),
                                  ("flatdense_d_3x3_n64", 2, 14, 64, 64, 3, 1, 1, False)], ids=lambda c: c[0])
def test_igemm_flat_window_dgrad(bcosk_lib, case):
    name, nb, h, cin, cout, k, plo, phi, f32 = case
    g = _gen(name)
    plan = _mini_plan(nb, 1)
    x = _rand_act(g, nb, h, h, cin, 1)
    w = torch.randn(cout, cin, k, k, generator=g) / math.sqrt(cin * k * k)
    oh = h + plo + phi - k + 1
    inv_norm = torch.rand(nb * oh * oh, generator=g) + 0.5
    _, rec = plan._conv_fwd(name, x, w, 1, plo, phi, bn=None, relu=True, want_mask=True, inv_norm=inv_norm,
                            kch=32 if cin == 32 else 64)
    rec.ghat = torch.zeros(nb, oh, oh, cout, dtype=plan.dt) if name.startswith("flatdense") \
        else plan._padded(nb, oh, oh, cout, k - 1 - plo, k - 1 - phi)
    rec.ghat_map = None
    rec.ghat.copy_(torch.randn(nb, oh, oh, cout, generator=g).to(plan.dt))
    M = nb * h * h
    yb = torch.zeros(nb, h, h, cin, dtype=torch.float32 if f32 else plan.dt)
    mul1 = None if f32 else (torch.rand(M, cin, generator=g) + 0.5).to(plan.gain_dt)
    add = None if f32 else _rand_act(g, nb, h, h, cin, 1).t
    out2 = None if f32 else torch.zeros(nb, h, h, cin, dtype=plan.dt)
    mask2 = None if f32 else torch.randint(-2**31, 2**31 - 1, (M, (cin + 31) // 32), generator=g, dtype=torch.int64).to(torch.int32)
    plan._dgrad(rec, y=yb, mul1=mul1, add=add, out2=out2, mask2=mask2, y_f32=f32, flat=True)
    assert plan.bwd_ops[-1].flat
    print(name, _run_and_compare(plan.bwd_ops))


@pytest.mark.parametrize("case", [("dc_3x3_s2", 2, 12, 64, 128, 3, 2, 1, 1), ("dc_3x3_s2_odd", 3, 14, 64, 64, 3, 2, 1, 1),
                                  ("dc_3x3_s2_planes2", 1, 8, 64, 64, 3, 2, 1, 2)], ids=lambda c: c[0])
def test_igemm_dgrad_parity_classes(bcosk_lib, case):
    """strided 3x3 data gradient as stride^2 parity-class launches over the dense gradient (side tensors by mapped row)"""
    name, nb, h, cin, cout, k, stride, pad, planes = case
    g = _gen(name)
    plan = _mini_plan(nb, planes)
    x = _rand_act(g, nb, h, h, cin, planes)
    w = torch.randn(cout, cin, k, k, generator=g) / math.sqrt(cin * k * k)
    _, rec = plan._conv_fwd(name, x, w, stride, pad, pad, bn=None, relu=True, want_mask=True)
    plan._alloc_ghat(rec, classes=True)
    assert rec.ghat_map is None and tuple(rec.ghat.shape[1:3]) == rec.out_hw
    oh, ow = rec.out_hw
    tmp = torch.zeros(nb, oh, ow, planes * cout, dtype=plan.dt)
    E._split_store(tmp, torch.randn(nb, oh, ow, cout, generator=g), planes)
    rec.ghat.copy_(tmp)
    M = nb * h * h
    yb = torch.zeros(nb, h, h, planes * cin, dtype=plan.dt)
    mul1 = (torch.rand(M, cin, generator=g) + 0.5).to(plan.gain_dt)
    plan._dgrad(rec, y=yb, mul1=mul1)
    assert len(plan.bwd_ops) == stride * stride and all(o.side_mapped for o in plan.bwd_ops)
    print(name, _run_and_compare(plan.bwd_ops, tol16=BF16_TOL if planes == 1 else 2e-4))
    # and against the zero-inserted single launch
    plan2 = _mini_plan(nb, planes)
    _, rec2 = plan2._conv_fwd(name, x, w, stride, pad, pad, bn=None, relu=True, want_mask=True)
    plan2._alloc_ghat(rec2)
    rec2.ghat[:, ::stride, ::stride][:, :oh, :ow] = tmp
    yb2 = torch.zeros_like(yb)
    plan2._dgrad(rec2, y=yb2, mul1=mul1)
    E.run(plan2.bwd_ops)
    a, b = E._join(yb, planes), E._join(yb2, planes)
    assert (a - b).abs().max() <= (2e-2 if planes == 1 else 1e-4) * b.abs().max()


def test_igemm_dgrad_strided_add_and_outmap(bcosk_lib):
    """conv1x1 data gradient that adds a half-resolution tensor and writes zero-inserted rows"""
    g = torch.Generator().manual_seed(11)
    nb, h, cin, cout = 2, 12, 64, 64
    plan = _mini_plan(nb, 1)
    x = _rand_act(g, nb, h, h, cin, 1)
    w = torch.randn(cout, cin, 1, 1, generator=g) / 8
    _, rec = plan._conv_fwd("c", x, w, 1, 0, 0, bn=None, relu=False)
    plan._alloc_ghat(rec)
    rec.ghat.copy_(torch.randn(nb, h, h, cout, generator=g).to(plan.dt))
    add = _rand_act(g, nb, h // 2, h // 2, cin, 1).t
    big = torch.zeros(nb, 2 * h, 2 * h, cin, dtype=plan.dt)
    plan._dgrad(rec, y=big, y_map=(0, 4 * h * h, 2 * 2 * h, 2), add=add, add_stride=2)
    print(_run_and_compare(plan.bwd_ops))
    assert float(big.abs().sum()) > 0


def test_a_tile_im2col(bcosk_lib):
    """what TMA im2col lands in shared memory == the emulator's gather (bit exact)"""
    g = torch.Generator().manual_seed(3)
    for (h, cin, k, stride, plo, phi, kch) in [(9, 64, 3, 1, 1, 1, 64), (9, 64, 3, 2, 1, 1, 64), (10, 32, 4, 1, 2, 1, 32),
                                                 (8, 128, 1, 2, 0, 0, 64)]:
        nb = 3
        plan = _mini_plan(nb, 1)
        x = _rand_act(g, nb, h, h, cin, 1)
        w = torch.randn(64, cin, k, k, generator=g)
        oh = (h + plo + phi - k) // stride + 1
        plan._conv_fwd("t", x, w, stride, plo, phi, bn=None, relu=False, kch=kch, inv_norm=torch.ones(nb * oh * oh))
        op = [o for o in plan.fwd_ops if isinstance(o, O.IgemmOp)][0]
        A = E.gather_a(op)                                   # [M, ktot]
        dop = U.to_device(op, "cuda")
        nchunks = op.ktot // kch
        m_tiles = (op.M + 127) // 128
        for tile_m in range(m_tiles):
            for chunk in sorted({0, 1 % nchunks, nchunks - 1}):
                out = torch.zeros(128, kch, dtype=torch.bfloat16, device="cuda")
                L.debug_a_tile(dop.params(), tile_m, chunk, out)
                torch.cuda.synchronize()
                exp = torch.zeros(128, kch)
                rows = min(128, op.M - tile_m * 128)
                exp[:rows] = A[tile_m * 128: tile_m * 128 + rows, chunk * kch:(chunk + 1) * kch]
                assert torch.equal(out.float().cpu(), exp), (h, cin, k, stride, kch, tile_m, chunk)


def test_persistent_sched_matches_per_tile(bcosk_lib):
    """same launch through the persistent (TMEM double-buffered) and the one-CTA-per-tile kernels"""
    nb, h, cin, cout = 4, 28, 128, 256
    outs = []
    for sched in (3, 2, 1):         # persistent in row-block order, persistent with tiles strided over the grid, one CTA per tile
        gg = torch.Generator().manual_seed(21)
        plan = _mini_plan(nb, 1)
        plan.light_k_iters = 18     # 18 K stages: 64-wide tiles (four column tiles), the only width with a persistent kernel
        x = _rand_act(gg, nb, h, h, cin, 1)
        w = torch.randn(cout, cin, 3, 3, generator=gg) / math.sqrt(cin * 9)
        plan.sd = {"bn.running_var": torch.rand(cout, generator=gg) + 0.5, "bn.weight": torch.rand(cout, generator=gg) + 0.5}
        res = _rand_act(gg, nb, h, h, cout, 1)
        y, rec = plan._conv_fwd("p", x, w, 1, 1, 1, bn="bn", relu=True, res=res, want_mask=True)
        op = plan.fwd_ops[-1]
        assert op.resolved_block_n() == 64
        op.sched = sched
        memo = {}
        dops = [U.to_device(o, "cuda", memo) for o in plan.fwd_ops]
        for o in dops:
            o.run()
        torch.cuda.synchronize()
        outs.append([t.cpu() for t in (dops[-1].y, dops[-1].gain, dops[-1].maskbits, dops[-1].sq_out)])
    for other in outs[:-1]:
        for k, (a, b) in enumerate(zip(other, outs[-1])):
            if k == 3:      # sums of squares: the persistent kernel adds two half-row partials (different rounding order)
                assert torch.allclose(a, b, rtol=1e-5, atol=0)
            else:
                assert torch.equal(a, b)


def test_light_and_late_input_variants_are_bit_identical(bcosk_lib):
    """the scheduling switches (CTAs per SM / ring slots, late input tile) only change how tiles are scheduled: every
    output must be bit-identical"""
    def build():
        g = torch.Generator().manual_seed(91)
        nb, h = 4, 16
        plan = _mini_plan(nb, 1)
        ops = []
        # forward 1x1, ONE K stage, residual (2-slot / 4-CTA variant) and TWO K stages (late input tile)
        for cin in (64, 128):
            x = _rand_act(g, nb, h, h, cin, 1)
            w = torch.randn(256, cin, 1, 1, generator=g) / math.sqrt(cin)
            plan.sd = {"bn.running_var": torch.rand(256, generator=g) + 0.5, "bn.weight": torch.rand(256, generator=g) + 0.5}
            res = _rand_act(g, nb, h, h, 256, 1)
            plan.fwd_ops.clear()
            _, rec = plan._conv_fwd(f"f{cin}", x, w, 1, 0, 0, bn="bn", relu=True, res=res, want_mask=True)
            ops += list(plan.fwd_ops)
        # 128-wide, long K loop, residual
        x = _rand_act(g, nb, h, h, 128, 1)
        w = torch.randn(256, 128, 3, 3, generator=g) / math.sqrt(128 * 9)
        res = _rand_act(g, nb, h, h, 256, 1)
        plan.fwd_ops.clear()
        _, rec3 = plan._conv_fwd("f3x3", x, w, 1, 1, 1, bn="bn", relu=True, res=res, want_mask=True)
        ops += list(plan.fwd_ops)
        # explain 1x1: one K stage, producer gain + extra gradient + second output + mask
        xe = _rand_act(g, nb, h, h, 256, 1)
        we = torch.randn(64, 256, 1, 1, generator=g) / 16
        plan.fwd_ops.clear()
        _, rece = plan._conv_fwd("e", xe, we, 1, 0, 0, bn=None, relu=True)
        plan._alloc_ghat(rece)
        rece.ghat.copy_(torch.randn(nb, h, h, 64, generator=g).to(plan.dt))
        M = nb * h * h
        plan._dgrad(rece, y=torch.zeros(nb, h, h, 256, dtype=plan.dt), mul1=(torch.rand(M, 256, generator=g) + 0.5).to(plan.gain_dt),
                    add=_rand_act(g, nb, h, h, 256, 1).t, out2=torch.zeros(nb, h, h, 256, dtype=plan.dt),
                    mask2=torch.randint(-2**31, 2**31 - 1, (M, 8), generator=g, dtype=torch.int64).to(torch.int32))
        # explain 3x3 128-wide with producer gain (late input tile, swapped output slots)
        plan._alloc_ghat(rec3)
        rec3.ghat.copy_(torch.randn(nb, h, h, 256, generator=g).to(plan.dt))
        plan._dgrad(rec3, y=torch.zeros(nb, h, h, 128, dtype=plan.dt), mul1=(torch.rand(M, 128, generator=g) + 0.5).to(plan.gain_dt))
        return ops + list(plan.bwd_ops)

    def run(light, late):
        prev = (bcosk_lib.bcosk_set_light(light), bcosk_lib.bcosk_set_late_input(late))
        try:
            memo = {}
            dops = [U.to_device(o, "cuda", memo) for o in build()]
            for o in dops:
                o.run()
            torch.cuda.synchronize()
            outs = []
            for o in dops:
                outs += [t.cpu() for t in (o.y, o.gain, o.maskbits, o.sq_out, o.out2) if t is not None]
            return outs
        finally:
            bcosk_lib.bcosk_set_light(prev[0]); bcosk_lib.bcosk_set_late_input(prev[1])

    ref_ops = build()
    print(_run_and_compare(ref_ops))                 # default switches against the emulator
    base = run(0, 0)                                 # 2 CTAs / SM everywhere, input tile parked in a ring slot
    for cfg in ((1, 0), (3, 2), (11, 2), (7, 1)):
        outs = run(*cfg)
        assert len(outs) == len(base)
        for a, b in zip(outs, base):
            assert torch.equal(a, b), cfg


@pytest.mark.parametrize("case", [("lazy_1x1", 1, False, 64), ("lazy_3x3", 3, False, 64), ("lazy_3x3_flat", 3, True, 64),
                                  ("lazy_1x1_n256", 1, False, 256)], ids=lambda c: c[0])
def test_gain_recomputed_from_relu_output(bcosk_lib, case):
    """gains that are not stored: forward writes 1/||patch|| (inv_norm_out), the consumer's explain epilogue multiplies by
    sqrt(y * inv) read from the producer's ReLU output (mul1_sqrt_scale)"""
    name, k, flat, cout = case
    g = _gen(name)
    nb, h, cin = 3, 12, 64
    plan = _mini_plan(nb, 1)
    plan.recompute_gain = True
    x = _rand_act(g, nb, h, h, cin, 1)
    wa = torch.randn(cout, cin, k, k, generator=g) / math.sqrt(cin * k * k)
    ya, ra = plan._conv_fwd("a", x, wa, 1, k // 2, k // 2, bn=None, relu=True, flat=flat)
    assert ra.gain is None and ra.gain_y is not None and ra.gain_inv is not None
    assert plan.fwd_ops[-1].gain is None and (flat or plan.fwd_ops[-1].inv_norm_out is not None)
    wb = torch.randn(64, cout, 3, 3, generator=g) / math.sqrt(cout * 9)
    yb, rb = plan._conv_fwd("b", ya, wb, 1, 1, 1, bn=None, relu=False)
    plan._alloc_ghat(rb)
    plan._alloc_ghat(ra)
    rb.ghat.copy_(torch.randn(nb, h, h, 64, generator=g).to(plan.dt))
    m1, m1s = plan._gain_of(ra)
    plan._dgrad(rb, y=ra.ghat, mul1=m1, mul1_sqrt_scale=m1s)
    assert plan.bwd_ops[-1].mul1_sqrt_scale is not None
    print(name, _run_and_compare(plan.fwd_ops + plan.bwd_ops))
    # and the same gradient with the gain stored the ordinary way
    plan2 = _mini_plan(nb, 1)
    plan2.recompute_gain = False
    ya2, ra2 = plan2._conv_fwd("a", x, wa, 1, k // 2, k // 2, bn=None, relu=True, flat=flat)
    yb2, rb2 = plan2._conv_fwd("b", ya2, wb, 1, 1, 1, bn=None, relu=False)
    plan2._alloc_ghat(rb2)
    plan2._alloc_ghat(ra2)
    rb2.ghat.copy_(rb.ghat)
    plan2._dgrad(rb2, y=ra2.ghat, mul1=ra2.gain)
    E.run(plan2.fwd_ops + plan2.bwd_ops)
    a, b = ra.ghat.float(), ra2.ghat.float()
    assert (a - b).abs().max() <= 2e-2 * b.abs().max()


@pytest.mark.parametrize("c,planes,k,st,pad", [(320, 2, 2, 2, 0), (448, 1, 2, 2, 0), (40, 2, 3, 2, 1), (8, 1, 2, 2, 0), (1056, 2, 2, 2, 0)])
def test_avgpool_any_channel_count(bcosk_lib, c, planes, k, st, pad):
    """pooling kernels for channel counts that are neither a power of two x 8 nor a multiple of 256 (DenseNet-169 / -201 transitions:
    320, 448, 896 channels)"""
    g = torch.Generator().manual_seed(c)
    nb, H = 2, 10
    dt = torch.bfloat16
    a = _rand_act(g, nb, H, H, c, planes)
    oh = (H + 2 * pad - k) // st + 1
    py = torch.zeros(nb, oh, oh, planes * c, dtype=dt)
    psq = torch.zeros(1, nb * oh * oh)
    ops = [O.AvgPoolFwdOp("pool", a.t, c, planes, k, st, pad, py, 1, psq)]
    gy = _rand_act(g, nb, oh, oh, c, planes).t
    gain = torch.rand(nb * H * H, c, generator=g).to(dt if planes == 1 else torch.float32)
    gx = torch.zeros(nb, H, H, planes * c, dtype=dt)
    ops.append(O.AvgPoolBwdMulOp("poolbwd", gy, c, planes, k, st, pad, gain, gx, 1))
    print(_run_and_compare(ops, tol16=BF16_TOL if planes == 1 else 2e-4))


@pytest.mark.parametrize("c,planes,W,k,st,pad", [(64, 2, 112, 3, 2, 1), (64, 3, 112, 3, 2, 1), (128, 2, 56, 2, 2, 0), (64, 1, 224, 3, 2, 1)])
def test_avgpool_long_rows_split_across_ctas(bcosk_lib, c, planes, W, k, st, pad):
    """row-staged pooling: rows whose k input rows exceed ~44 KB of shared memory are shared by two or three CTAs"""
    g = torch.Generator().manual_seed(W + c)
    nb, H = 1, 10
    a = _rand_act(g, nb, H, W, c, planes)
    oh, ow = (H + 2 * pad - k) // st + 1, (W + 2 * pad - k) // st + 1
    py = torch.zeros(nb, oh, ow, planes * c, dtype=torch.bfloat16)
    psq = torch.zeros(1, nb * oh * ow)
    print(_run_and_compare([O.AvgPoolFwdOp("pool", a.t, c, planes, k, st, pad, py, 1, psq)], tol16=BF16_TOL if planes == 1 else 2e-4))


def test_elementwise_kernels(bcosk_lib):
    g = torch.Generator().manual_seed(5)
    nb, S = 3, 32
    for planes in (1, 2, 3):
        dt = torch.bfloat16
        x = torch.rand(nb, 3, S, S, generator=g)
        x6 = torch.cat([x, 1 - x], 1).contiguous()
        mean = (0.485, 0.456, 0.406, 0.515, 0.544, 0.594)
        istd = tuple(1 / s for s in (0.229, 0.224, 0.225, 0.229, 0.224, 0.225))
        out = torch.zeros(nb, S // 2, S // 2, planes * 32, dtype=dt)
        sq = torch.zeros(1, nb * S * S)
        ops = [O.InputPrepOp("prep", x6, mean, istd, out, 32, planes, 1, sq)]
        inv = torch.zeros(nb * 16 * 16)
        ops.append(O.PatchNormOp("norm7", sq, 1, nb, S, S, 7, 2, 3, 1e-6, 0.0, inv, 16, 16))
        a = _rand_act(g, nb, 16, 16, 64, planes)
        py = torch.zeros(nb, 8, 8, planes * 64, dtype=dt)
        psq = torch.zeros(1, nb * 64)
        ops.append(O.AvgPoolFwdOp("pool", a.t, 64, planes, 3, 2, 1, py, 1, psq))
        gy = _rand_act(g, nb, 8, 8, 64, planes).t
        gain = (torch.rand(nb * 256, 64, generator=g)).to(dt if planes == 1 else torch.float32)
        gx = torch.zeros(nb, 16, 16, planes * 64, dtype=dt)
        ops.append(O.AvgPoolBwdMulOp("poolbwd", gy, 64, planes, 3, 2, 1, gain, gx, 1))
        if planes == 1:     # the same two kernels writing the interior view of a zero-bordered buffer
            plan = _mini_plan(nb, 1)
            outp = plan._padded(nb, S // 2, S // 2, 32, 2, 1)
            ops.append(O.InputPrepOp("prep_padded", x6, mean, istd, outp, 32, 1, 1, torch.zeros(1, nb * S * S)))
            gxp = plan._padded(nb, 16, 16, 64, 1, 2)
            ops.append(O.AvgPoolBwdMulOp("poolbwd_padded", gy, 64, 1, 3, 2, 1, gain, gxp, 1))
            # the multiplier recomputed as sqrt(y * scale) from a ReLU output
            ops.append(O.AvgPoolBwdMulOp("poolbwd_lazy_gain", gy, 64, 1, 3, 2, 1, gain, torch.zeros(nb, 16, 16, 64, dtype=dt), 1,
                                         torch.rand(nb * 256, generator=g) + 0.5))
        fc = torch.randn(nb * 49, 1000, generator=g)
        logits = torch.zeros(nb, 1000)
        pred = torch.zeros(nb, dtype=torch.int32)
        ops.append(O.GapLogitsOp("gap", fc, nb, 49, 1000, 1.0, -6.9, logits, pred))
        gfc = torch.rand(nb * 49, 1000, generator=g).to(dt if planes == 1 else torch.float32)
        wfc = torch.randn(1000, 128, generator=g)
        mul1 = torch.rand(nb * 49, 128, generator=g).to(dt if planes == 1 else torch.float32)
        mask2 = torch.randint(-2**31, 2**31 - 1, (nb * 49, 4), generator=g, dtype=torch.int64).to(torch.int32)
        o1 = torch.zeros(nb * 49, planes * 128, dtype=dt)
        o2 = torch.zeros(nb * 49, planes * 128, dtype=dt)
        tgt = torch.tensor([3, 999, 500], dtype=torch.int32)
        ops.append(O.FcSeedOp("seed", tgt, gfc, wfc, nb, 49, 1000, 128, 1.0, 4.0, mul1, o1, mask2, o2, planes, 1))
        g0 = torch.randn(nb, S // 2, S // 2, 32, generator=g)
        cmap = torch.zeros(nb, S, S)
        grad6 = torch.zeros(nb, 6, S, S)
        ops.append(O.ContribMapOp("cmap", g0, x6, 32, istd, 0.25, cmap, grad6))
        print(planes, _run_and_compare(ops, tol16=BF16_TOL if planes == 1 else 2e-4))


@pytest.mark.parametrize("u8", [False, True], ids=["x6_f32", "rgb_u8"])
def test_explanation_rgba(bcosk_lib, u8):
    """device gradient_to_image for a batch (colour, alpha, 15x15 box filter, per-image 99.5 percentile by radix select)
    against the oracle's restatement of bcos/common.py:387-436"""
    g = torch.Generator().manual_seed(77)
    nb, S = 3, 64
    x3 = torch.rand(nb, 3, S, S, generator=g)
    x = (x3 * 255).round().to(torch.uint8) if u8 else torch.cat([x3, 1 - x3], 1).contiguous()
    grad6 = torch.randn(nb, 6, S, S, generator=g) * torch.rand(nb, 1, S, S, generator=g)
    for smooth, pct in ((15, 99.5), (0, 90.0), (3, 100.0)):
        op = O.ExplanationImageOp("rgba", grad6, x, smooth, pct, torch.zeros(2 * nb * S * S + nb), torch.zeros(nb, S, S, 4))
        print(smooth, pct, _run_and_compare([op], tol32=2e-5))
