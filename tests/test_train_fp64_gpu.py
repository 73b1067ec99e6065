"""The fine-tuning step's kernels against fp64 references computed from the same 16-bit operands the kernels read.

Products of two 16-bit values are exact in fp32, so every bound below covers only accumulation and the final rounding, and each
is derived from the kernel's summation structure (written next to it), not fitted to a measurement.  The measured error is printed
beside its bound on `REPORT` lines.

  1. `bcosk_wgrad` at every geometry the ResNet-50 and DenseNet-121 training plans launch (collected from the plans, so the test
     follows them), explicit split-K settings, the bench-size stem and layer1 launches, and negative controls that the bound
     must reject.
  2. A small bottleneck ResNet step (the stem, four stages with a downsample each, fp32 classifier) against fp64 autograd, and the
     plan's AGC + AdamW update against an fp64 step from its own gradients.
  3. The whole-model AGC + AdamW kernel, the device-side Adam step counter and the packed-operand refresh over three steps, with
     the real unit / gather tables of ResNet-50 and DenseNet-121.  A CPU-only check that the AGC units tile the master buffer.
  4. Batch-statistics BN (`bnu_stats_nhwc` -> `bnu_finalize`, `dense_slice_stats`) at bench row counts, channel means far from 0.
  5. The train-kernel flags the plans use: fp16, fp32 data gradients, the fp32 classifier, absent gb / tn / g_y, grad_combine,
     and sumpool_transpose at every geometry the plans' patch-norm paths launch.
"""
import functools
import math
import zlib

import pytest
import torch

import bcos_oracle as OR
from bcos_b200 import _lib as L
from bcos_b200.engine import ResNetTrainPlan
from bcos_b200.engine import resnet as RS
from bcos_b200.engine.train import DenseNetTrainPlan, FnOp, WgradOp
from bcos_b200.utils import synth

DT = {"bf16": torch.bfloat16, "fp16": torch.float16}
U16 = {"bf16": 2.0 ** -8, "fp16": 2.0 ** -11}        # unit roundoff of one round-to-nearest 16-bit store
U16_ABS = {"bf16": 2.0 ** -134, "fp16": 2.0 ** -25}  # ... and its absolute floor (half the subnormal spacing)
U32 = 2.0 ** -24
NBLK = 296                                           # TrainPlanBase.red_blocks: rows of partial sums of the per-channel reductions
KP = 64                                              # pixels per K stage of bcosk_wgrad


def _gen(name, device="cuda"):
    g = torch.Generator(device=device)
    g.manual_seed(zlib.crc32(name.encode()))
    return g


def _rel(a, b):
    return float((a.double() - b.double()).norm() / (b.double().norm() + 1e-300))


def _cos(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float(torch.dot(a, b) / (a.norm() * b.norm() + 1e-300))


def _f32(*v):
    """the fp32 values the kernels receive for these host floats"""
    return [float(t) for t in torch.tensor(v, dtype=torch.float32).double()]


def _ulp(w):
    a = w.abs().float()
    return (torch.nextafter(a, torch.full_like(a, math.inf)) - a).double()


@functools.lru_cache(maxsize=None)
def _cpu_plan(arch, size, batch):
    if arch.startswith("resnet"):
        sd = synth.synth_state_dict(OR.resnet_state_shapes(arch), 0)
        return ResNetTrainPlan(arch, sd, batch, device="cpu", image_size=size)
    sd = synth.synth_state_dict(OR.densenet_state_shapes(arch), 0)
    return DenseNetTrainPlan(arch, sd, batch, device="cpu", image_size=size)


# ================================================================================================ 1. weight gradient
def _wgrad_geometries():
    """Distinct `WgradOp` geometries of the ResNet-50 and DenseNet-121 plans at 224^2, batch 2: [(key, op)]."""
    out = {}
    for arch in ("resnet50", "densenet121"):
        for op in _cpu_plan(arch, 224, 2).bwd_ops:
            if isinstance(op, WgradOp):
                f = op.fwd
                key = (tuple(f.a.shape), f.n, tuple(f.taps), f.stride, f.lo, f.up, f.kch, f.chunks_per_tap, op.g.shape[-1])
                out.setdefault(key, (arch, op))
    return list(out.values())


def _split_geom(p, split_k, sms):
    """bcosk_wgrad's host heuristic (csrc/bcosk_wgrad.cu): (pixels per CTA K_cta, CTAs along the pixel axis, 64-pixel blocks)."""
    bn = 128 if (p.kch == 64 and p.chunks_per_tap % 2 == 0) else p.kch
    col_tiles = p.num_taps * p.chunks_per_tap // (bn // p.kch)
    blocks_total = -(-(p.a_nb * p.op * p.oq) // KP)
    o_tiles = -(-p.n // 128)
    split = split_k
    if split <= 0:
        split = -(-4 * sms // (o_tiles * col_tiles))
        split = max(1, min(split, max(blocks_total // 8, 1)))
    blocks_per = -(-blocks_total // split)
    split = -(-blocks_total // blocks_per)
    return blocks_per * KP, split, blocks_total


def _wgrad_ref(x, g, p, drop_from=None):
    """dw[o, t, c] = sum_m g[m, o] x[img, p s_h + lo_h + off_h[t], q s_w + lo_w + off_w[t], c] in fp64 (zero outside the image
    and for c >= a_c), and A = the same sum of |g| |x|.  `drop_from`: pixels m >= drop_from left out."""
    nb, h, w, c = x.shape
    kw = p.kch * p.chunks_per_tap
    xd = torch.zeros(nb, h, w, kw, dtype=torch.float64, device=x.device)
    xd[..., :c] = x.double()
    gd = g[:, :p.n].double()
    if drop_from is not None:
        gd = gd.clone()
        gd[drop_from:] = 0
    ref = torch.empty(p.n, p.num_taps, kw, dtype=torch.float64, device=x.device)
    A = torch.empty_like(ref)
    dev = x.device
    for t in range(p.num_taps):
        ih = torch.arange(p.op, device=dev) * p.stride_h + p.lo_h + p.tap_off_h[t]
        iw = torch.arange(p.oq, device=dev) * p.stride_w + p.lo_w + p.tap_off_w[t]
        mask = (((ih >= 0) & (ih < h))[:, None] & ((iw >= 0) & (iw < w))[None, :]).to(torch.float64)
        X = xd[:, ih.clamp(0, h - 1)][:, :, iw.clamp(0, w - 1)] * mask[None, :, :, None]
        X = X.reshape(-1, kw)
        ref[:, t] = gd.t() @ X
        if drop_from is None:
            A[:, t] = gd.abs().t() @ X.abs()
    return ref.reshape(p.n, -1), A.reshape(p.n, -1)


def _wgrad_launch(op, x, g, dtype, split_k, prefill):
    """`op`'s launch geometry over fresh operands x [nb, h, w, a_c] and g [M, g_ld], accumulating into a copy of `prefill`."""
    p = op.params()
    p.x, p.a_nb = x.data_ptr(), x.shape[0]
    p.g = g.data_ptr()
    dw = prefill.clone()
    p.dw = dw.data_ptr()
    p.dtype = L.DTYPE_CODE[dtype]
    p.split_k = split_k
    L.wgrad(p)
    torch.cuda.synchronize()
    return dw, p


def _wgrad_operands(op, nb, dtype, tag, g_pos=False):
    f = op.fwd
    gen = _gen(tag)
    shape = (nb,) + tuple(f.a.shape[1:])
    x = torch.rand(shape, device="cuda", generator=gen).to(DT[dtype])           # >= 0, like a ReLU / image input
    M = nb * f.op * f.oq
    g = torch.randn(M, op.g.shape[-1], device="cuda", generator=gen)
    g = (g.abs() if g_pos else g).to(DT[dtype])
    return x, g


def _bound(K_cta, split, A, P):
    """Per element: K_cta products accumulated in one TMEM accumulator (truncating adds: 2^-23 per add, relative to the running
    sum, itself <= A), then `split` partial tiles and the prefilled value added with round-to-nearest fp32 reductions."""
    return (K_cta + split + 2) * 2.0 ** -23 * (A + P.double().abs())


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
def test_wgrad_every_plan_geometry_within_fp64_bound(bcosk_lib, dtype):
    """Every distinct `bcosk_wgrad` geometry of the ResNet-50 / DenseNet-121 training plans: the default split and split_k 1, 3
    and all blocks, each within its own per-element bound; columns c >= a_c bit-exactly untouched; dw accumulated onto a prefilled
    pattern.  Negative controls: references without the last 64-pixel block, with two taps swapped, with the last o-tile's units
    shifted by one, must each break the bound somewhere."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    geoms = _wgrad_geometries()
    bad = []
    for gi, (arch, op) in enumerate(geoms):
        f = op.fwd
        nb, a_c = f.a.shape[0], f.a.shape[3]
        x, g = _wgrad_operands(op, nb, dtype, f"wgrad{gi}{dtype}")
        p0 = op.params()
        p0.a_nb = nb
        ref, A = _wgrad_ref(x, g, p0)
        gen = _gen(f"prefill{gi}{dtype}")
        P = (torch.randn(ref.shape, device="cuda", generator=gen) * 1e-3 * float(A.max())).float()
        P[P == 0] = 1.0
        kw = f.kch * f.chunks_per_tap
        bt = _split_geom(p0, 0, sms)[2]
        line = []
        for split_k in (0, 1, 3, bt):
            dw, p = _wgrad_launch(op, x, g, dtype, split_k, P)
            K_cta, split, _ = _split_geom(p, split_k, sms)
            bound = _bound(K_cta, split, A, P)
            err = (dw.double() - P.double() - ref)
            worst = float((err.abs() / bound).max())
            desc = (f"{arch}:{op.name} x{tuple(x.shape)} n={f.n} taps={len(f.taps)} s={f.stride} kch={f.kch} cpt={f.chunks_per_tap} "
                    f"split_k={split_k}")
            line.append(f"split {split} K_cta {K_cta}: {worst:.2e}")
            if not worst <= 1.0:
                bad.append(f"{desc}: {worst:.3e}")
            if kw > a_c:
                pad = (dw.view(f.n, len(f.taps), kw)[..., a_c:], P.view(f.n, len(f.taps), kw)[..., a_c:])
                if not torch.equal(pad[0].view(torch.int32), pad[1].view(torch.int32)):
                    bad.append(f"{desc}: columns c >= a_c = {a_c} changed")
            if split_k != 0:
                continue
            # negative controls against the same kernel output and bound
            got = dw.double() - P.double()
            M = x.shape[0] * f.op * f.oq
            drop, _ = _wgrad_ref(x, g, p0, drop_from=(-(-M // KP) - 1) * KP)
            controls = {"last pixel block dropped": drop}
            if len(f.taps) > 1:
                sw = ref.view(f.n, len(f.taps), kw).clone()
                sw[:, [0, 1]] = sw[:, [1, 0]]
                controls["taps 0 and 1 swapped"] = sw.view(f.n, -1)
            o0 = 128 * ((f.n - 1) // 128)
            sh = ref.clone()
            sh[o0:] = torch.roll(ref[o0:], 1, dims=0)
            controls["last o-tile shifted by one unit"] = sh
            for what, r in controls.items():
                if not bool(((got - r).abs() > bound).any()):
                    bad.append(f"{desc}: negative control '{what}' passes the bound")
        print(f"REPORT wgrad {dtype} {arch}:{op.name} x{tuple(x.shape)} n={f.n} taps={len(f.taps)} s={f.stride} kch={f.kch} "
              f"cpt={f.chunks_per_tap}: max |err|/bound " + ", ".join(line))
    print(f"REPORT wgrad {dtype}: {len(geoms)} geometries x 4 splits")
    assert not bad, "\n".join(bad)


def _bench_op(name):
    return [o for o in _cpu_plan("resnet50", 224, 2).bwd_ops if isinstance(o, WgradOp) and o.name == name][0]


@pytest.mark.gpu
@pytest.mark.parametrize("name,g_pos", [("stem.wgrad", False), ("stem.wgrad", True), ("model.layer1.0.conv1.wgrad", False)])
def test_wgrad_bench_size_accumulation(bcosk_lib, name, g_pos):
    """ResNet-50's stem (M = 64 x 112 x 112 pixels, 16 taps, kch 32) and layer1's 1x1 64 -> 64 at the benchmark's batch 64, bf16,
    default split.  Reports the largest error in units of 2^-24 K_cta A (A = sum |g| |x|) and its sign bias; g >= 0 with x >= 0 is
    the case in which the truncating accumulation cannot cancel."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    op = _bench_op(name)
    nb = 64
    x, g = _wgrad_operands(op, nb, "bf16", f"bench{name}{g_pos}", g_pos=g_pos)
    P = torch.zeros(op.fwd.n, op.fwd.ktot, device="cuda")
    dw, p = _wgrad_launch(op, x, g, "bf16", 0, P)
    ref, A = _wgrad_ref(x, g, p)
    K_cta, split, _ = _split_geom(p, 0, sms)
    err = dw.double() - ref
    unit = K_cta * U32 * A
    r = err / unit
    nz = err != 0
    worst = float((err.abs() / _bound(K_cta, split, A, P)).max())
    print(f"REPORT wgrad bench {name} g>=0={g_pos} M={nb * p.op * p.oq} split={split} K_cta={K_cta}: max |err| = {float(r.abs().max()):.3e} "
          f"x 2^-24 K_cta A, mean err = {float(r.mean()):+.3e} x 2^-24 K_cta A, {float((err[nz] < 0).double().mean()):.3f} of the "
          f"nonzero errors negative; max |err|/bound {worst:.3e}")
    assert worst <= 1.0


# ================================================================================================ 2. small bottleneck step
def _small_arch(monkeypatch):
    arch = "resnet_bneck_1111_t"
    cfg = ("bottleneck", [1, 1, 1, 1])
    monkeypatch.setitem(RS.RESNET_ARCH, arch, cfg)
    monkeypatch.setitem(OR.RESNET_ARCH, arch, cfg)
    return arch


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,loss_scale", [("fp16", 65536.0), ("bf16", 1.0)])
def test_small_bottleneck_step_matches_fp64_autograd(bcosk_lib, monkeypatch, dtype, loss_scale):
    """A bottleneck ResNet with one block per stage (stem, four downsamples, strided 3x3 and strided 1x1 data gradients,
    grad_combine, the pool backward, the fp32 classifier) at 64^2, batch 4, against fp64 autograd with the same fp16-rounded conv
    weights and fp64-calibrated BN.

    How far 16-bit operands may move a gradient follows from this net's own sensitivity to rounding: the reference's fp32 gradients
    are 6e-6 .. 8.8e-6 (relative, per tensor; the stem's BN weight the largest) away from its fp64 ones.  fp16 operands round
    2^13 x coarser than fp32, so they are expected to move the gradients by up to ~0.07; each tensor must stay within twice what
    its own fp32 gap predicts, and within 0.03 where that is larger.  (A per-tensor floor of cosine 0.9995 / relative error 0.03,
    as for the small DenseNet whose gradients are far less sensitive, is not supported here: the stem's BN weight measured 0.086 in
    fp16 on a B200; every tensor measured 1.19 - 1.28 x its prediction, so the error tracks the net's sensitivity.)  bf16 rounds 2^16 x coarser than fp32; the linear prediction exceeds 1, so bf16 is held to the loss and to
    a cosine floor of 0.95 (measured minimum 0.974, again the stem's BN weight).
    Then the AGC + AdamW update against an fp64 step from the plan's own gradients and pre-step master weights: per element within
    2 ulp(w) + 1e-5 lr."""
    arch = _small_arch(monkeypatch)
    S, nb = 64, 4
    sd = synth.synth_state_dict(OR.resnet_state_shapes(arch), 0)
    imgs = synth.synth_images_u8(nb, S, 5)
    labels = torch.arange(nb) * 71 % 1000
    sd16 = {k: (v.to(torch.float16).float() if k.endswith(".linear.weight") else v) for k, v in sd.items()}
    sd64 = {k: (v.double() if v.is_floating_point() else v) for k, v in sd16.items()}
    x64 = synth.to_bcos_input(imgs).double()
    om = OR.OracleResNet(arch, sd64)
    om.calibrate_bn(x64)
    ref = OR.train_step_reference(om, x64, labels)
    sd32 = {k: (v.float() if v.is_floating_point() else v) for k, v in sd16.items()}
    om32 = OR.OracleResNet(arch, sd32)
    om32.calibrate_bn(x64.float())
    gap = {k: _rel(v, ref["grads"][k]) for k, v in OR.train_step_reference(om32, x64.float(), labels)["grads"].items()}
    sd_plan = {k: (v.float() if v.is_floating_point() else v) for k, v in sd64.items()}      # calibrated running variances
    plan = ResNetTrainPlan(arch, sd_plan, nb, dtype=dtype, device="cuda", image_size=S, loss_scale=loss_scale)
    w0 = plan.w_flat.clone()
    loss = plan.train_step(torch.from_numpy(imgs), labels)
    torch.cuda.synchronize()
    loss_rel = abs(float(loss) - float(ref["loss"])) / float(ref["loss"])
    g = plan.gradients()
    assert set(g) == set(ref["grads"])
    cos = {k: _cos(g[k].cpu(), r) for k, r in ref["grads"].items()}
    rel = {k: _rel(g[k].cpu(), r) for k, r in ref["grads"].items()}
    worst = min(cos, key=cos.get)
    new = plan.state_dict()
    rv = {k: _rel(new[k].cpu(), v) for k, v in ref["running_var"].items()}
    for k in sorted(rel, key=rel.get):
        print(f"REPORT small bottleneck {dtype} {k}: cos {cos[k]:.6f} rel {rel[k]:.3e} (fp32 gap {gap[k]:.2e}, "
              f"rel / (gap 2^13) {rel[k] / (gap[k] * 2 ** 13):.2f})")
    print(f"REPORT small bottleneck {dtype}: loss rel {loss_rel:.2e}; min cos {cos[worst]:.6f} ({worst}); max rel "
          f"{max(rel.values()):.3e} ({max(rel, key=rel.get)}); running_var max rel {max(rv.values()):.2e}")
    if dtype == "fp16":
        assert loss_rel <= 2e-4
        over = {k: r for k, r in rel.items() if r > max(0.03, 2 * 2 ** 13 * gap[k])}
        assert not over, over
        assert max(rv.values()) < 2e-3
    else:
        assert loss_rel <= 1e-3
        assert cos[worst] >= 0.95
    # the update, from the plan's own gradients and pre-step weights
    h = dict(zip(plan.hyper, _f32(*plan.hyper.values())))
    st = plan.adam_state.cpu().double()
    assert float(st[0]) == 1.0
    worst_u = 0.0
    for key, w, off in plan._w_items:
        wp = w0[off:off + w.numel()].view(w.shape).double().cpu()
        gc = OR.adaptive_clip_grad(wp, g[key].double().cpu(), h["clip"], h["agc_eps"])
        m = (1 - h["beta1"]) * gc
        v = (1 - h["beta2"]) * gc * gc
        want = wp - h["lr"] * h["wd"] * wp - h["lr"] * (m / st[1]) / ((v / st[2]).sqrt() + h["eps"])
        got = new[key].double().cpu()
        tol = 2 * _ulp(want) + 1e-5 * h["lr"]
        q = float(((got - want).abs() / tol).max())
        worst_u = max(worst_u, q)
        assert q <= 1.0, key
    print(f"REPORT small bottleneck {dtype} update: max |w - w_fp64| / (2 ulp + 1e-5 lr) = {worst_u:.3f}")


# ================================================================================================ 3. whole-model optimizer
def _sorted_units(plan):
    off = plan.unit_off.cpu().long()
    cols = plan.unit_cols.cpu().long()
    order = torch.argsort(off)
    return off[order], cols[order], order


@pytest.mark.parametrize("arch", ["resnet50", "densenet121"])
def test_agc_units_tile_master_weights(arch):
    """Without a GPU: the AGC units of a plan tile its fp32 master buffer exactly (no gap, no overlap), and every unit is one
    output row of a state-dict conv / classifier weight (the 7x7 stem: 6 x 49 = 294 columns, not the s2d operand's width) or a
    whole 1-D BN weight."""
    plan = _cpu_plan(arch, 64, 2)
    off, cols, _ = _sorted_units(plan)
    assert int(off[0]) == 0 and bool((cols > 0).all())
    assert torch.equal(off[1:], off[:-1] + cols[:-1])
    assert int(off[-1] + cols[-1]) == plan.w_flat.numel()
    want = []
    for key, w, o in plan._w_items:
        if w.ndim >= 2:
            c = w.numel() // w.shape[0]
            want += [(o + i * c, c) for i in range(w.shape[0])]
        else:
            want.append((o, w.numel()))
    assert sorted(want) == list(zip(off.tolist(), cols.tolist()))
    stem = [k for k, _, _ in plan._w_items if k.endswith(".linear.weight")][0]
    sw = [(w, o) for k, w, o in plan._w_items if k == stem][0]
    assert tuple(sw[0].shape[1:]) == (6, 7, 7) and (sw[1], 294) in want


@pytest.mark.gpu
@pytest.mark.parametrize("arch", ["resnet50", "densenet121"])
def test_whole_model_agc_adamw_three_steps_match_fp64(bcosk_lib, arch):
    """Three steps of `adam_state_step` + `agc_adamw_multi` over the plan's real tables (gidx, unit_off, unit_cols), weight decay
    0.05, grad_scale 1 / (2 x 65536).  Each step: fresh seeded gradients scaled per unit so that about half the units clip (1.1 -
    3 x the threshold) and half do not (0.2 - 0.9 x), with the unclipped gradients 10^3 smaller and the clipped ones 10^3 larger
    than on the step before.  Reference: fp64 `adaptive_clip_grad` per state-dict tensor, then AdamW.  After every step, w / m / v
    element by element, the step counter, and the packed-operand refresh in both dtypes bit-exactly (plus an odd-length entry).

    Bounds: the clip factor comes from fp32 sums of at most 4608 / 256 + 5 + 8 = 31 rounded terms per unit norm, so its relative
    error is below 2e-6 (taken as 4e-6); m and v inherit it (v twice) plus a few fp32 roundings: 1e-5 of their running absolute
    sums.  u = m^ / (sqrt(v^) + eps) inherits m's absolute error and half of v's relative error; w then gets lr x that plus two fp32
    roundings (the decay and the update) per step, accumulated over the steps."""
    S, nb = 64, 2
    if arch.startswith("resnet"):
        sd = synth.synth_state_dict(OR.resnet_state_shapes(arch), 0)
        plan = ResNetTrainPlan(arch, sd, nb, device="cuda", image_size=S)
    else:
        sd = synth.synth_state_dict(OR.densenet_state_shapes(arch), 0)
        plan = DenseNetTrainPlan(arch, sd, nb, device="cuda", image_size=S)
    hyper = (0.9, 0.999, 1e-8, 1e-4, 0.05, 0.01, 1e-3)
    b1, b2, eps, lr, wd, clip, agc_eps = _f32(*hyper)             # the reference uses the fp32 values the kernel receives
    gscale = 1.0 / (2 * 65536.0)
    off, cols, order = _sorted_units(plan)
    n_w, U = plan.w_flat.numel(), off.numel()
    elem_unit = torch.repeat_interleave(order, cols).cuda()       # unit of every master element (the units tile the buffer)
    gidx = plan.gidx.long()
    w64 = plan.w_flat.double()
    m64 = torch.zeros_like(w64)
    v64 = torch.zeros_like(w64)
    mabs = torch.zeros_like(w64)
    tol_w = torch.zeros_like(w64)
    gen = _gen(f"agc{arch}")
    for step in range(3):
        # gradients: per unit, a target ratio to the clipping threshold
        nw = torch.zeros(U, dtype=torch.float64, device="cuda").index_add_(0, elem_unit, w64 * w64).sqrt()
        max_norm = nw.clamp(min=agc_eps) * clip
        clipped = torch.rand(U, device="cuda", generator=gen) < 0.5
        u = torch.rand(U, device="cuda", generator=gen).double()
        ratio = torch.where(clipped, (1.1 + 1.9 * u) * 1e3 ** step, (0.2 + 0.7 * u) * 1e-3 ** step)
        gm = torch.randn(n_w, device="cuda", generator=gen).double()
        gn = torch.zeros(U, dtype=torch.float64, device="cuda").index_add_(0, elem_unit, gm * gm).sqrt()
        gm = gm * (ratio * max_norm / gn)[elem_unit]
        plan.g_flat.zero_()
        plan.g_flat[gidx] = (gm / gscale).float()
        gk = plan.g_flat[gidx].double() * gscale                   # what the kernel reads, exactly
        L.adam_state_step(plan.adam_state, b1, b2)
        L.agc_adamw_multi(plan.w_flat, plan.g_flat, plan.gidx, plan.m_flat, plan.v_flat, plan.unit_off, plan.unit_cols, U, gscale,
                          lr, b1, b2, eps, wd, clip, agc_eps, plan.adam_state)
        torch.cuda.synchronize()
        t = step + 1
        st = plan.adam_state.cpu().double()
        assert float(st[0]) == t
        bc = [1 - b1 ** t, 1 - b2 ** t]
        for i in (1, 2):                                           # powf: a few ulp of beta^t (< 1), then one exact subtraction
            assert abs(float(st[i]) - bc[i - 1]) <= 4 * U32, (t, i, float(st[i]), bc[i - 1])
        # fp64 reference, AGC per state-dict tensor (the unit definition of agc.py, not the plan's table)
        gc = torch.empty_like(w64)
        for key, w, o in plan._w_items:
            sl = slice(o, o + w.numel())
            gc[sl] = OR.adaptive_clip_grad(w64[sl].view(w.shape), gk[sl].view(w.shape), clip, agc_eps).reshape(-1)
        frac_clipped = float(clipped.double().mean())
        bc1, bc2 = float(st[1]), float(st[2])                      # the device's bias corrections (checked above)
        m64 = b1 * m64 + (1 - b1) * gc
        v64 = b2 * v64 + (1 - b2) * gc * gc
        mabs = b1 * mabs + (1 - b1) * gc.abs()
        den = (v64 / bc2).sqrt() + eps
        upd = (m64 / bc1) / den
        w64 = w64 - lr * wd * w64 - lr * upd
        tol_m = 1e-5 * mabs
        tol_v = 1e-5 * v64
        tol_u = (tol_m / bc1) / den + upd.abs() * (0.5e-5 + 8 * U32)
        tol_w = tol_w + lr * tol_u + 2 * _ulp(w64)
        q = {name: float(((got.double() - want).abs() / (tol + 1e-300)).max())
             for name, got, want, tol in (("w", plan.w_flat, w64, tol_w), ("m", plan.m_flat, m64, tol_m), ("v", plan.v_flat, v64, tol_v))}
        print(f"REPORT agc_adamw_multi {arch} step {t}: {U} units, {frac_clipped:.2f} clipped; max err/bound " +
              " ".join(f"{k} {v:.3f}" for k, v in q.items()))
        assert 0.4 < frac_clipped < 0.6
        assert max(q.values()) <= 1.0, q
        # operand refresh: every packed operand, and an odd-length entry (the tail element), in both dtypes
        for dtype, dt in DT.items():
            idx_syn = torch.randint(-1, n_w, (1001,), device="cuda", generator=gen, dtype=torch.int32)
            entries = [(idx, torch.full(idx.shape, -7.0, dtype=dt, device="cuda")) for _, idx in plan.packs]
            entries.append((idx_syn, torch.full((1001,), -7.0, dtype=dt, device="cuda")))
            table = torch.tensor([[i.data_ptr(), o.data_ptr(), i.numel()] for i, o in entries], dtype=torch.int64, device="cuda")
            L.gather_cast_multi(plan.w_flat, table, len(entries), max(i.numel() for i, _ in entries), L.DTYPE_CODE[dtype])
            torch.cuda.synchronize()
            for i, o in entries:
                want = torch.where(i >= 0, plan.w_flat[i.clamp(min=0).long()], torch.zeros((), device="cuda")).to(dt)
                assert torch.equal(o.view(torch.int16), want.view(torch.int16)), (dtype, i.numel())


# ================================================================================================ 4. batch statistics
def _stats_bounds(xd, rows, c, nblk):
    """Bounds of bnu_stats -> finalize (and dense_slice_stats): each thread sums r = ceil(rows / (nblk RP)) rows in fp32 (one
    rounding per add / fma), its block adds RP such partials in fp32, the partials are summed in fp64 (exact enough to ignore):
    |d sum x| <= (r + RP) 2^-24 sum |x|, |d sum x^2| <= (r + RP) 2^-24 sum x^2.  Then mean = s1 / M, var = s2 / M - mean^2."""
    G = c // 8
    RP = max(1, 256 // G)
    r = -(-rows // (nblk * RP))
    k = (r + RP + 1) * U32
    mean = xd.mean(0)
    var = ((xd - mean) ** 2).mean(0)
    e1 = k * xd.abs().sum(0) / rows
    e2 = k * (xd * xd).sum(0) / rows
    d_mean = e1 + U32 * mean.abs()
    d_var = e2 + (2 * mean.abs() + e1) * e1 + 1e-14 * (xd * xd).mean(0)
    return mean, var, d_mean, d_var, r, RP


def _offset_rows(rows, c, dtype, tag):
    """rows x c 16-bit values, unit standard deviation, channel means 0, 2 and 10 standard deviations (thirds of the channels)"""
    gen = _gen(tag)
    mu = torch.tensor([0.0, 2.0, 10.0], device="cuda")[torch.arange(c, device="cuda") % 3]
    return (torch.randn(rows, c, device="cuda", generator=gen) + mu).to(DT[dtype]), mu


@pytest.mark.gpu
@pytest.mark.parametrize("rows,c", [(64 * 112 * 112, 64), (64 * 28 * 28, 512), (3136, 2048)])
@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
def test_batch_stats_at_bench_rows_within_derived_bound(bcosk_lib, rows, c, dtype):
    """bnu_stats_nhwc -> bnu_finalize at the bench stem (64 x 112^2 rows, 64 channels), layer2's conv3 output and layer4 at batch 64
    (3136 x 2048): mean, rstd, alpha and the running-variance EMA per channel within the bound propagated from the summation."""
    x, mu = _offset_rows(rows, c, dtype, f"bnstats{rows}{c}{dtype}")
    xd = x.double()
    mean, var, d_mean, d_var, r, RP = _stats_bounds(xd, rows, c, NBLK)
    gen = _gen(f"bnw{rows}{c}{dtype}")
    w = torch.rand(c, device="cuda", generator=gen) + 0.5
    rv0 = torch.rand(c, device="cuda", generator=gen) + 0.5
    part = torch.empty(NBLK, 2 * c, device="cuda")
    L.bnu_stats_nhwc(x, rows, c, L.DTYPE_CODE[dtype], part)
    outs = [torch.empty(c, device="cuda") for _ in range(3)]
    rv = rv0.clone()
    eps, mom = 1e-5, 0.1
    L.bnu_finalize(part, rows, c, w, eps, mom, rv, *outs)
    torch.cuda.synchronize()
    alpha, m_k, rstd = (o.double() for o in outs)
    rstd_ref = 1 / (var + eps).sqrt()
    d_rstd = 0.5 * 1.01 * rstd_ref ** 3 * d_var + U32 * rstd_ref
    rv_ref = (1 - mom) * rv0.double() + mom * var
    d_rv = mom * (d_var + U32 * var) + 3 * U32 * rv_ref
    checks = {"mean": ((m_k - mean).abs(), d_mean), "rstd": ((rstd - rstd_ref).abs(), d_rstd),
              "alpha": ((alpha - w.double() * rstd_ref).abs(), w.double() * d_rstd + 2 * U32 * w.double() * rstd_ref),
              "running_var": ((rv.double() - rv_ref).abs(), d_rv)}
    for off in (0.0, 2.0, 10.0):
        sel = mu == off
        print(f"REPORT bn stats {dtype} rows={rows} c={c} (r={r}, RP={RP}) channel mean {off:g} sd: " + " ".join(
            f"{k} err/bound {float((e[sel] / b[sel]).max()):.3f}" for k, (e, b) in checks.items()) +
            f"; var rel err {float(((1 / rstd[sel] ** 2 - eps) / var[sel] - 1).abs().max()):.1e}")
    for k, (e, b) in checks.items():
        assert bool((e <= b).all()), k


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
def test_dense_slice_stats_largest_prefix_within_derived_bound(bcosk_lib, dtype):
    """dense_slice_stats over DenseNet-121's widest prefix (block 3's 1024 channels at 14^2, batch 64), in a wider feature tensor"""
    rows, c, ld = 64 * 14 * 14, 1024, 1024 + 64
    F, mu = _offset_rows(rows, ld, dtype, f"dense{dtype}")
    xd = F.double()[:, :c]
    mean, var, d_mean, d_var, r, RP = _stats_bounds(xd, rows, c, NBLK)
    part = torch.empty(NBLK, 2 * c, device="cuda")
    stats = [torch.full((ld,), -7.0, device="cuda") for _ in range(3)]
    eps = 1e-5
    L.dense_slice_stats(F, rows, ld, 0, c, eps, part, *stats, L.DTYPE_CODE[dtype])
    torch.cuda.synchronize()
    m_k, v_k, r_k = (s[:c].double() for s in stats)
    rstd_ref = 1 / (var + eps).sqrt()
    checks = {"mean": ((m_k - mean).abs(), d_mean), "var": ((v_k - var).abs(), d_var + U32 * var),
              "rstd": ((r_k - rstd_ref).abs(), 0.5 * 1.01 * rstd_ref ** 3 * d_var + U32 * rstd_ref)}
    print(f"REPORT dense slice stats {dtype} rows={rows} c={c} (r={r}, RP={RP}): " +
          " ".join(f"{k} err/bound {float((e / b).max()):.3f}" for k, (e, b) in checks.items()))
    for k, (e, b) in checks.items():
        assert bool((e <= b).all()), k
    assert all(bool((s[c:] == -7.0).all()) for s in stats)


# ================================================================================================ 5. train-kernel flags
def _bwd_case(rows, c, dtype, tag, ga_f32, out_f32):
    gen = _gen(tag)
    dt = DT[dtype]
    r = lambda *s: torch.randn(*s, device="cuda", generator=gen)              # noqa: E731
    ga = r(rows, c) * 0.01
    ga = ga if ga_f32 else ga.to(dt)
    gb = (r(rows, c) * 0.01).to(dt)
    xpost = r(rows, c).clamp(min=0).to(dt) if not out_f32 else None
    tn = r(rows) * 0.01
    out = r(rows, c) * 2 + 0.3
    out = out if out_f32 else out.to(dt)
    s = (torch.rand(rows, c, device="cuda", generator=gen) + 0.1).to(dt)
    inv = torch.rand(rows, device="cuda", generator=gen) + 0.5
    alpha = torch.rand(c, device="cuda", generator=gen) + 0.5
    mean = r(c) * 0.1
    rstd = torch.rand(c, device="cuda", generator=gen) + 0.5
    w = torch.rand(c, device="cuda", generator=gen) + 0.5
    return ga, gb, xpost, tn, out, s, inv, alpha, mean, rstd, w


def _gy_ref(ga, gb, xpost, tn, relu):
    """g_y = (ga + gb + xpost tn[row]) [xpost > 0] in fp64, and the sum of the magnitudes of its terms"""
    g = ga.double()
    gabs = g.abs()
    if gb is not None:
        g = g + gb.double()
        gabs = gabs + gb.double().abs()
    if xpost is not None and tn is not None:
        t = xpost.double() * tn.double()[:, None]
        g = g + t
        gabs = gabs + t.abs()
    if xpost is not None and relu:
        keep = xpost.double() > 0
        g, gabs = g * keep, gabs * keep
    return g, gabs


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [
    dict(bn=True, relu=True, gb=True, tn=True, gy=True, c=64),                     # a block's last conv (all inputs)
    dict(bn=True, relu=True, gb=False, tn=True, gy=False, c=2048),                  # an inner conv
    dict(bn=True, relu=True, gb=True, tn=False, gy=False, c=256),                   # tn absent
    dict(bn=True, relu=False, gb=False, tn=False, gy=False, c=512),                 # the downsample: no ReLU, no patch-norm path
    dict(bn=True, relu=True, gb=False, tn=True, gy=False, c=128, ga_f32=True),     # the DenseNet's fp32 data gradients
    dict(bn=False, relu=False, gb=False, tn=False, gy=False, c=1000, out_f32=True),  # the classifier
])
@pytest.mark.parametrize("dtype", ["fp16", "bf16"])
def test_train_backward_flags_match_fp64(bcosk_lib, flags, dtype):
    """train_bwd_reduce -> bnu_bwd_finalize -> train_bwd_apply against fp64 restatements of the header's formulas, per element.
    Bounds: g_y is at most three fp32 operations (2^-24 each of the sum of its terms' magnitudes), g_out one fma and one product
    more; 16-bit outputs add one rounding (U16).  The reduction S: r = ceil(rows / (nblk RP)) fmas per thread, RP partials per
    block, fp64 across blocks.  gnT: 8 G / lanes fmas per lane and log2(lanes) shuffle adds, then two products."""
    rows, c = 3001, flags["c"]
    ga_f32, out_f32 = flags.get("ga_f32", False), flags.get("out_f32", False)
    relu = flags["relu"]
    dtc = L.DTYPE_CODE[dtype]
    ga, gb, xpost, tn, out, s, inv, alpha, mean, rstd, w = _bwd_case(rows, c, dtype, f"bwd{c}{dtype}{ga_f32}{out_f32}", ga_f32, out_f32)
    gb = gb if flags["gb"] else None
    tn = tn if flags["tn"] else None
    xpost = xpost if (relu or tn is not None) else None
    gy, gabs = _gy_ref(ga, gb, xpost, tn, relu)
    od = out.double()
    e_gy = 3 * U32 * gabs
    if flags["bn"]:
        G = c // 8
        RP = max(1, 256 // G)
        r = -(-rows // (NBLK * RP))
        part = torch.empty(NBLK, c, device="cuda")
        L.train_bwd_reduce(ga, ga_f32, gb, xpost, tn, relu, out, out_f32, rows, c, part, dtc)
        kcoef, gw, s_out = (torch.empty(c, device="cuda") for _ in range(3))
        L.bnu_bwd_finalize(part, rstd, w, rows, c, kcoef, gw, s_out)
        torch.cuda.synchronize()
        S = (gy * od).sum(0)
        dS = (r + RP + 1) * U32 * (gabs * od.abs()).sum(0) + (e_gy * od.abs()).sum(0)
        rd, wd_ = rstd.double(), w.double()
        k_ref = -rd ** 3 * wd_ * S / rows
        q_red = {"S": float(((s_out.double() - S).abs() / (dS + U32 * S.abs())).max()),
                 "kcoef": float(((kcoef.double() - k_ref).abs() / (rd ** 3 * wd_ * dS / rows * 1.001 + U32 * k_ref.abs())).max()),
                 "g_weight": float(((gw.double() - S * rd).abs() / (rd * dS * 1.001 + U32 * (S * rd).abs())).max())}
        k_in = kcoef
    else:
        q_red = {}
        k_in = None
    glin = torch.empty(rows, c, dtype=DT[dtype], device="cuda")
    gnt = torch.empty(rows, device="cuda")
    gy_out = torch.empty(rows, c, dtype=DT[dtype], device="cuda") if flags["gy"] else None
    a_in, m_in = (alpha, mean) if flags["bn"] else (None, None)
    L.train_bwd_apply(ga, ga_f32, gb, xpost, tn, relu, out, out_f32, s, a_in, k_in, m_in, inv, rows, c, glin, gnt, gy_out, dtc)
    torch.cuda.synchronize()
    if flags["bn"]:
        kd = k_in.double()
        go = gy * alpha.double() + (od - mean.double()) * kd
        e_go = e_gy * alpha.double() + 3 * U32 * (gabs * alpha.double() + ((od - mean.double()) * kd).abs())
        go_abs = gabs * alpha.double() + ((od - mean.double()) * kd).abs()
    else:
        go, e_go, go_abs = gy, e_gy, gabs
    sd_ = s.double()
    gl_ref = 2 * go * sd_
    b_gl = U16[dtype] * gl_ref.abs() + 2 * sd_ * (e_go + U32 * go_abs) * (1 + U16[dtype]) + U16_ABS[dtype]
    G = c // 8
    lanes = min(G, 32)
    n_acc = 8 * -(-G // lanes) + int(math.log2(lanes)) + 3
    invd = inv.double()
    gnt_ref = -(go * od).sum(1) * invd ** 2
    b_gnt = (n_acc * U32 * (go_abs * od.abs()).sum(1) + (e_go * od.abs()).sum(1)) * invd ** 2
    q = dict(q_red)
    q["g_lin"] = float(((glin.double() - gl_ref).abs() / (b_gl + 1e-300)).max())
    q["gnT"] = float(((gnt.double() - gnt_ref).abs() / (b_gnt + 1e-300)).max())
    if gy_out is not None:
        q["g_y"] = float(((gy_out.double() - gy).abs() / (U16[dtype] * gy.abs() + e_gy * (1 + U16[dtype]) + U16_ABS[dtype])).max())
    print(f"REPORT train bwd {dtype} {flags}: max err/bound " + " ".join(f"{k} {v:.3f}" for k, v in q.items()))
    assert max(q.values()) <= 1.0, q


@pytest.mark.gpu
@pytest.mark.parametrize("with_gb,with_tn", [(True, True), (False, True), (True, False), (False, False)])
@pytest.mark.parametrize("dtype", ["fp16", "bf16"])
def test_grad_combine_matches_fp64(bcosk_lib, dtype, with_gb, with_tn):
    """out = ga + gb + x tn[row] rounded once to 16 bits (at most three fp32 operations before it)"""
    rows, c = 2 * 56 * 56 + 5, 64
    ga, gb, x, tn, *_ = _bwd_case(rows, c, dtype, f"comb{dtype}{with_gb}{with_tn}", False, False)
    gb = gb if with_gb else None
    tn = tn if with_tn else None
    out = torch.empty(rows, c, dtype=DT[dtype], device="cuda")
    L.grad_combine(ga, gb, x, tn, rows, c, out, L.DTYPE_CODE[dtype])
    torch.cuda.synchronize()
    ref, gabs = _gy_ref(ga, gb, x if tn is not None else None, tn, False)
    b = U16[dtype] * ref.abs() + 3 * U32 * gabs * (1 + U16[dtype]) + U16_ABS[dtype]
    q = float(((out.double() - ref).abs() / (b + 1e-300)).max())
    print(f"REPORT grad_combine {dtype} gb={with_gb} tn={with_tn}: max err/bound {q:.3f}")
    assert q <= 1.0


def _normpath_geometries():
    """(nb, h, w, k, stride, pad, op, oq) of every sumpool_transpose launch the plans' patch-norm paths emit"""
    out = set()
    for arch in ("resnet50", "densenet121"):
        for op in _cpu_plan(arch, 224, 2).bwd_ops:
            if isinstance(op, FnOp) and op.name.endswith(".normpath"):
                cl = dict(zip(op.fn.__code__.co_freevars, (c.cell_contents for c in op.fn.__closure__)))
                out.add((cl["self"].nb, cl["h"], cl["w"], cl["k"], cl["s"], cl["pad"], cl["oh"], cl["ow"]))
    return sorted(out)


@pytest.mark.gpu
def test_sumpool_transpose_plan_geometries_match_fp64(bcosk_lib):
    """tn (+)= the sum of gnT over the windows that cover each input pixel, against an fp64 conv_transpose2d with a ones kernel,
    at every geometry the plans launch, with accumulate 0 and 1.  At most k^2 fp32 adds (+1 for accumulate)."""
    geoms = _normpath_geometries()
    assert geoms
    for nb, h, w, k, s, pad, oh, ow in geoms:
        gen = _gen(f"sumpool{h}{k}{s}{pad}")
        gnt = torch.randn(nb * oh * ow, device="cuda", generator=gen)
        prev = torch.randn(nb * h * w, device="cuda", generator=gen)
        one = torch.ones(1, 1, k, k, dtype=torch.float64, device="cuda")
        full = torch.nn.functional.conv_transpose2d(gnt.double().view(nb, 1, oh, ow), one, stride=s)
        fa = torch.nn.functional.conv_transpose2d(gnt.double().abs().view(nb, 1, oh, ow), one, stride=s)
        ref, A = (torch.zeros(nb, 1, h + pad, w + pad, dtype=torch.float64, device="cuda") for _ in range(2))
        hh, ww = min(full.shape[2], h + pad), min(full.shape[3], w + pad)
        ref[:, :, :hh, :ww], A[:, :, :hh, :ww] = full[:, :, :hh, :ww], fa[:, :, :hh, :ww]
        ref, A = ref[:, 0, pad:, pad:].reshape(-1), A[:, 0, pad:, pad:].reshape(-1)
        worst = []
        for acc in (0, 1):
            tn = prev.clone()
            L.sumpool_transpose(gnt, nb, h, w, k, s, pad, oh, ow, acc, tn)
            torch.cuda.synchronize()
            want = ref + (prev.double() if acc else 0)
            b = (k * k + acc) * U32 * (A + (prev.double().abs() if acc else 0)) + 1e-300
            worst.append(float(((tn.double() - want).abs() / b).max()))
        print(f"REPORT sumpool_transpose nb={nb} {h}x{w} k={k} s={s} pad={pad} -> {oh}x{ow}: max err/bound {worst[0]:.3f} / {worst[1]:.3f} (accumulate 0 / 1)")
        assert max(worst) <= 1.0
