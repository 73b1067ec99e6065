"""-m gpu: the CLIP ResNet fine-tuning step (CLIPResNetTrainPlan, engine/clip_train.py).

The new kernels against torch fp64 (average-pool backward fused with the consumers' terms, softmax backward); the attention-pool
head's backward at its real size against fp64 autograd of `OracleCLIPResNet.attnpool` with q and k in the graph; a small CLIP
ResNet step against fp64 autograd with the same rounded weights; a whole CLIP RN50 step against the fp32 oracle.

Conditioning of the whole-step configuration (CLIP RN50, 64^2, batch 8, synthetic seed-0 weights, images seed 5, a cosine
distillation loss to fixed unit targets): see `test_clip_rn50_train_step_matches_oracle`, which measures the oracle's own fp32 vs
fp64 gap per tensor and prints it next to the plan's cosines.
"""
import json
import math
import os
import subprocess
import sys
import zlib

import pytest
import torch
import torch.nn.functional as F

import bcos_oracle as OR
from bcos_b200 import _lib as L
from bcos_b200.engine import CLIPResNetPlan, CLIPResNetTrainPlan
from bcos_b200.utils import synth

pytestmark = pytest.mark.gpu
DT = {"bf16": torch.bfloat16, "fp16": torch.float16}
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EPS32 = 2.0 ** -24
# measured on a B200: min cosine 0.99836 and max relative error 5.8e-2, both on layer2.0's bn1 weight (whose fp32 gap, 9.9e-6, is the
# largest of this net); the three mutations of the head / pool backward drop the minimum to 0.0, 0.895 and 0.913
SMALL_MIN_COS, SMALL_MAX_REL = 0.997, 0.08


def _rel(a, b):
    return float((a.double() - b.double()).norm() / (b.double().norm() + 1e-300))


def _cos(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float(torch.dot(a, b) / (a.norm() * b.norm() + 1e-300))


def _gen(name):
    g = torch.Generator(device="cuda")
    g.manual_seed(zlib.crc32(name.encode()))
    return g


# ---------------------------------------------------------------------------------------------------------------- kernels
# (nb, h, w, c): a block pool (layer2.0 at 224^2: 56 -> 28, 128 channels), a downsample pool (256 channels), the stem pool
# (112 -> 56 at 224^2, 64 channels; here 30 x 31: the last row / column lie past the last full window)
POOL_CASES = [(2, 56, 56, 128), (3, 14, 14, 256), (2, 30, 31, 64)]


@pytest.mark.parametrize("nb,h,w,c", POOL_CASES)
@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("ga_f32", [False, True])
@pytest.mark.parametrize("accumulate", [False, True])
def test_pool_bwd_norm_matches_torch(bcosk_lib, nb, h, w, c, dtype, ga_f32, accumulate):
    """gx (+)= AvgPool2d(2) backward of (ga + gb + xp * tn): one 16-bit rounding of the fp64 value (of the sum with the old gx)"""
    k = 2
    op, oq = h // k, w // k
    dt, dtc = DT[dtype], L.DTYPE_CODE[dtype]
    g = _gen(f"pool{nb}{h}{w}{c}{dtype}{ga_f32}{accumulate}")
    rows = nb * op * oq
    ga = torch.randn(rows, c, device="cuda", generator=g) * 0.01
    ga = ga if ga_f32 else ga.to(dt)
    gb = (torch.randn(rows, c, device="cuda", generator=g) * 0.01).to(dt)
    xp = torch.randn(rows, c, device="cuda", generator=g).clamp(min=0).to(dt)
    tn = torch.randn(rows, device="cuda", generator=g) * 0.01
    gx0 = (torch.randn(nb, h, w, c, device="cuda", generator=g) * 0.01).to(dt)
    pooled = (ga.double() + gb.double() + xp.double() * tn.double()[:, None]).view(nb, op, oq, c) / (k * k)
    want = torch.zeros(nb, h, w, c, dtype=torch.float64, device="cuda")
    want[:, :op * k, :oq * k] = pooled.repeat_interleave(k, 1).repeat_interleave(k, 2)
    if accumulate:
        want += gx0.double()
    ulp = 2.0 ** (-8 if dtype == "bf16" else -11)
    sub = 0.0 if dtype == "bf16" else 2.0 ** -25           # half the spacing of fp16's subnormals (below 2^-14)
    for with_gb in (True, False):
        gx = gx0.clone()
        L.pool_bwd_norm(ga, ga_f32, gb if with_gb else None, xp, tn, nb, h, w, c, k, accumulate, gx, dtc)
        torch.cuda.synchronize()
        ref = want
        if not with_gb:
            ref = want.clone()
            ref[:, :op * k, :oq * k] -= (gb.double().view(nb, op, oq, c) / (k * k)).repeat_interleave(k, 1).repeat_interleave(k, 2)
        err = (gx.double() - ref).abs()
        # one rounding of the result; the fp32 sum of at most four terms before it
        assert bool((err <= ulp * ref.abs() + sub + 8 * EPS32 * (ref.abs() + 1e-3)).all()), float(err.max())
        gx2 = gx0.clone()
        L.pool_bwd_norm(ga, ga_f32, gb if with_gb else None, xp, tn, nb, h, w, c, k, accumulate, gx2, dtc)
        assert torch.equal(gx2, gx)


@pytest.mark.parametrize("n", [5, 50, 197])
def test_softmax_bwd_matches_fp64(bcosk_lib, n):
    """ds = p (dp - sum p dp): per element within n 2^-24 (|p dp| + p sum |p dp|); in place (ds aliases dp) too; bit-reproducible"""
    rows = 8 * 32 + 3
    g = _gen(f"smb{n}")
    p = torch.softmax(torch.randn(rows, n, device="cuda", generator=g) * 3, dim=1)
    dp = torch.randn(rows, n, device="cuda", generator=g)
    p64, d64 = p.double(), dp.double()
    want = p64 * (d64 - (p64 * d64).sum(1, keepdim=True))
    bound = (n + 2) * EPS32 * (p64 * d64.abs() + p64 * (p64 * d64.abs()).sum(1, keepdim=True))
    ds = torch.empty_like(dp)
    L.softmax_bwd(p, dp, rows, n, ds)
    torch.cuda.synchronize()
    assert bool(((ds.double() - want).abs() <= bound).all())
    ds2 = torch.empty_like(dp)
    L.softmax_bwd(p, dp, rows, n, ds2)
    assert torch.equal(ds2, ds)
    inplace = dp.clone()
    L.softmax_bwd(p, inplace, rows, n, inplace)
    torch.cuda.synchronize()
    assert torch.equal(inplace, ds)


# ---------------------------------------------------------------------------------------------------------------- head
def _head_fp64(tok, wq, wk, wv, wc, heads, g_emb):
    """The commuted head and its backward (engine/clip_train.py docstring) in fp64, with the magnitudes Sum |a||b| of the last
    product of every gradient."""
    nb, T, C = tok.shape
    dh = C // heads
    s = dh ** -0.5
    x0 = tok[:, 0]
    q = s * x0 @ wq.t()
    qt = torch.einsum("bhd,hdc->bhc", q.view(nb, heads, dh), wk.view(heads, dh, C))
    p = torch.softmax(torch.einsum("bhc,btc->bht", qt, tok), -1)
    xbar = torch.einsum("bht,btc->bhc", p, tok)
    o = torch.einsum("hdc,bhc->bhd", wv.view(heads, dh, C), xbar).reshape(nb, C)
    g_o = g_emb @ wc
    g_xbar = torch.einsum("bhd,hdc->bhc", g_o.view(nb, heads, dh), wv.view(heads, dh, C))
    dp = torch.einsum("bhc,btc->bht", g_xbar, tok)
    ds = p * (dp - (p * dp).sum(-1, keepdim=True))
    g_qt = torch.einsum("bht,btc->bhc", ds, tok)
    g_q = torch.einsum("bhc,hdc->bhd", g_qt, wk.view(heads, dh, C)).reshape(nb, C)
    A = abs
    mag = {
        "model.attnpool.c_proj.linear.weight": A(g_emb).t() @ A(o),
        "model.attnpool.v_proj.weight": torch.einsum("bhd,bhc->hdc", A(g_o).view(nb, heads, dh), A(xbar)).reshape(C, C),
        "model.attnpool.k_proj.weight": torch.einsum("bhd,bhc->hdc", A(q).view(nb, heads, dh), A(g_qt)).reshape(C, C),
        "model.attnpool.q_proj.weight": s * A(g_q).t() @ A(x0),
    }
    g_tok_mag = torch.einsum("bht,bhc->btc", p, A(g_xbar)) + torch.einsum("bht,bhc->btc", A(ds), A(qt))
    g_tok_mag[:, 0] += s * A(g_q) @ A(wq)
    return mag, g_tok_mag


def test_head_backward_matches_fp64_autograd(bcosk_lib):
    """C = 2048, 32 heads, 50 tokens (7 x 7 trunk output), batch 4: the head's launches of a plan on fp32 tokens against fp64
    autograd of `OracleCLIPResNet.attnpool` (q and k NOT detached).  Every gradient element is within
    k 2^-24 Sum |a||b| of its last product, k = 3 C + 2 T + nb (the length of the fp32 chain in front of it)."""
    nb, S = 4, 224
    layers = (1, 1, 1, 1)
    sd = synth.synth_state_dict(OR.clip_rn_state_shapes(layers), 0)
    plan = CLIPResNetTrainPlan(sd, nb, layers=layers, dtype="bf16", device="cuda", image_size=S)
    C, H, T = plan.trunk_out.c, plan.heads, plan.tokens.shape[1]
    assert (C, H, T) == (2048, 32, 50)
    g = _gen("head")
    x = torch.randn(nb, C, 7, 7, device="cuda", generator=g, dtype=torch.float64).clamp(min=0)
    pix = x.flatten(2).transpose(1, 2)
    tok64 = torch.cat([pix.mean(1, keepdim=True), pix], 1)
    plan.tokens.copy_(tok64.float())
    g_emb = torch.randn(nb, plan.emb.shape[1], device="cuda", generator=g) * 1e-3
    plan.g_emb.copy_(g_emb)
    for op in plan.fwd_ops + plan.bwd_ops:
        if op.name.startswith("attnpool.") and op.name not in ("attnpool.tokens", "attnpool.seed"):
            op.run()
    torch.cuda.synchronize()
    keys = ["model.attnpool.q_proj.weight", "model.attnpool.k_proj.weight", "model.attnpool.v_proj.weight",
            "model.attnpool.c_proj.linear.weight"]
    sd64 = {k: sd[k].double().cuda().requires_grad_(True) for k in keys}
    om = OR.OracleCLIPResNet(sd64, layers=layers)
    xg = x.clone().requires_grad_(True)
    with torch.enable_grad():
        emb = om.attnpool(xg, detach=False)
        grads = torch.autograd.grad(emb, [sd64[k] for k in keys] + [xg], g_emb.double())
    ref = dict(zip(keys + ["x"], grads))
    assert _rel(plan.emb, emb.detach()) < 1e-5
    wq, wk, wv, wc = (sd[k].double().cuda() for k in keys)
    mag, g_tok_mag = _head_fp64(tok64, wq, wk, wv, wc, H, g_emb.double())
    kf = 3 * C + 2 * T + nb
    got = plan.gradients()
    worst = {}
    for k in keys:
        err = (got[k].double() - ref[k]).abs()
        bound = kf * EPS32 * mag[k]
        worst[k] = float((err / (bound + 1e-300)).max())
        assert bool((err <= bound).all()), (k, worst[k])
    # d pixels = d tokens[pixel] + d tokens[mean] / npix
    gt = plan.g_tokens.double()
    g_pix = gt[:, 1:] + gt[:, :1] / (T - 1)
    ref_pix = ref["x"].flatten(2).transpose(1, 2)
    mag_pix = g_tok_mag[:, 1:] + g_tok_mag[:, :1] / (T - 1)
    err = (g_pix - ref_pix).abs()
    worst["tokens"] = float((err / (kf * EPS32 * mag_pix + 1e-300)).max())
    print("REPORT head backward: max err / bound " + ", ".join(f"{k} {v:.3f}" for k, v in worst.items()))
    assert bool((err <= kf * EPS32 * mag_pix).all())


# ---------------------------------------------------------------------------------------------------------------- whole steps
def _targets(nb, d):
    return F.normalize(torch.randn(nb, d, generator=torch.Generator().manual_seed(11)), dim=1)


def _cos_loss(targets):
    def loss_fn(emb):
        return (1 - F.cosine_similarity(emb, targets.to(emb.device, emb.dtype), dim=1)).mean()
    return loss_fn


def clip_train_reference(model, x6, loss_fn, momentum=0.1):
    """One train-mode step of the oracle (autograd of every trainable weight: conv / BN weights and the head's q, k, v, c_proj);
    returns loss, embedding, gradients and the updated running variances."""
    keys = [k for k, v in model.sd.items() if v.is_floating_point() and k.endswith(".weight")]
    saved = dict(model.sd)
    params = {k: model.sd[k].detach().clone().requires_grad_(True) for k in keys}
    model.sd = {**{k: (v.clone() if torch.is_tensor(v) else v) for k, v in saved.items()}, **params}
    model.training, model.momentum = True, momentum
    try:
        with torch.enable_grad():
            emb = model.forward(x6)
            loss = loss_fn(emb)
            grads = torch.autograd.grad(loss, [params[k] for k in keys])
        running = {k: v.detach().clone() for k, v in model.sd.items() if k.endswith("running_var")}
    finally:
        model.training, model.momentum = False, 0.1
        model.sd = saved
    return {"loss": loss.detach(), "emb": emb.detach(), "grads": dict(zip(keys, grads)), "running_var": running}


def test_small_clip_resnet_step_matches_fp64_autograd(bcosk_lib):
    """layers (1, 1, 1, 1), 64^2, batch 4, fp16 with loss scaling, the conv weights rounded to fp16 on both sides: every weight
    gradient (stem, the four blocks with their anti-aliasing pools and downsample pools, the head's q / k / v / c_proj), the
    running variances and the loss against fp64 autograd of the oracle in train mode."""
    layers, S, nb = (1, 1, 1, 1), 64, 4
    sd = synth.synth_state_dict(OR.clip_rn_state_shapes(layers), 0)
    sd16 = {k: (v.to(torch.float16).float() if (k.endswith(".linear.weight") and v.ndim == 4) else v) for k, v in sd.items()}
    sd64 = {k: (v.double() if v.is_floating_point() else v) for k, v in sd16.items()}
    imgs = synth.synth_images_u8(nb, S, 5)
    x64 = synth.to_bcos_input(imgs).double()
    om = OR.OracleCLIPResNet(sd64, layers=layers)
    om.calibrate_bn(x64)
    tg = _targets(nb, 1024)
    ref = clip_train_reference(om, x64, _cos_loss(tg.double()))
    sd_plan = {k: (v.float() if v.is_floating_point() else v) for k, v in om.sd.items()}
    ref32 = clip_train_reference(OR.OracleCLIPResNet(dict(sd_plan), layers=layers), x64.float(), _cos_loss(tg))
    gap = {k: _rel(r, ref["grads"][k]) for k, r in ref32["grads"].items()}
    plan = CLIPResNetTrainPlan(sd_plan, nb, layers=layers, dtype="fp16", device="cuda", image_size=S, loss_scale=1024.0)
    loss = plan.train_step(torch.from_numpy(imgs), _cos_loss(tg))
    torch.cuda.synchronize()
    assert abs(float(loss) - float(ref["loss"])) <= 1e-3 * float(ref["loss"])
    g = plan.gradients()
    assert set(g) == set(ref["grads"])
    cos = {k: _cos(g[k].cpu(), r) for k, r in ref["grads"].items()}
    rel = {k: _rel(g[k].cpu(), r) for k, r in ref["grads"].items()}
    worst = min(cos, key=cos.get)
    print(f"REPORT small clip resnet fp16: min cos {cos[worst]:.6f} ({worst}, fp32 gap {gap[worst]:.1e}) max rel {max(rel.values()):.3e} "
          f"({max(rel, key=rel.get)}); max fp32 gap {max(gap.values()):.1e} ({max(gap, key=gap.get)})")
    assert cos[worst] >= SMALL_MIN_COS and max(rel.values()) < SMALL_MAX_REL
    new = plan.state_dict()
    rv = {k: _rel(new[k].cpu(), v) for k, v in ref["running_var"].items()}
    print(f"REPORT small clip resnet running_var: max rel {max(rv.values()):.3e}")
    assert set(rv) == {k for k in sd if k.endswith("running_var")} and max(rv.values()) < 2e-3


def _rn50_case():
    S, nb = 64, 8
    sd = synth.synth_state_dict(OR.clip_rn_state_shapes(), 0)
    imgs = synth.synth_images_u8(nb, S, 5)
    return S, nb, sd, imgs, _targets(nb, 1024)


# measured on a B200: fp16 every tensor >= 0.9239, the head's >= 0.9668 (median 0.952); bf16 the head's >= 0.405, median 0.308
@pytest.mark.parametrize("dtype,loss_scale,min_cos,head_cos,median_cos", [("fp16", 1024.0, 0.9, 0.95, 0.93), ("bf16", 1.0, None, 0.35, 0.25)])
def test_clip_rn50_train_step_matches_oracle(bcosk_lib, dtype, loss_scale, min_cos, head_cos, median_cos):
    """CLIP RN50 at 64^2, batch 8 against the fp32 oracle: loss, gradient keys, per-tensor cosines (printed with the oracle's own
    fp32 vs fp64 gap), running variances, the first AdamW step, the operand refresh, a second step; the updated state dict loads
    into CLIPResNetPlan and embeds like the oracle with the updated weights.

    This train-mode step is badly conditioned: the oracle's own fp32 gradients are up to 1.2e-3 (typically 5e-4) from fp64, 60 times
    the DenseNet-121 step's gap, and even the head's gradients depend on the whole train-mode forward (the embedding).  One 16-bit
    rounding is 2^13 (fp16) / 2^16 (bf16) times coarser than fp32, so the floors are set below the measured minimums: per tensor in
    fp16; in bf16 only the head's tensors and the median mean anything.  The small-network test above is the precise check (fp32 gap
    1e-5, cosines >= 0.998)."""
    S, nb, sd, imgs, tg = _rn50_case()
    x6 = synth.to_bcos_input(imgs)
    om = OR.OracleCLIPResNet(sd)
    om.calibrate_bn(x6)
    sd_cal = dict(om.sd)
    ref = clip_train_reference(om, x6, _cos_loss(tg))
    sd64 = {k: (v.double() if v.is_floating_point() else v) for k, v in sd_cal.items()}
    ref64 = clip_train_reference(OR.OracleCLIPResNet(sd64), x6.double(), _cos_loss(tg.double()))
    gap = {k: _rel(r, ref64["grads"][k]) for k, r in ref["grads"].items()}
    plan = CLIPResNetTrainPlan(sd_cal, nb, dtype=dtype, device="cuda", image_size=S, loss_scale=loss_scale)
    loss = plan.train_step(torch.from_numpy(imgs), _cos_loss(tg))
    torch.cuda.synchronize()
    assert abs(float(loss) - float(ref["loss"])) <= 2e-3 * float(ref["loss"])
    g = plan.gradients()
    assert set(g) == set(ref["grads"]) and all(math.isfinite(float(v.abs().sum())) for v in g.values())
    cos = {k: _cos(g[k].cpu(), r) for k, r in ref["grads"].items()}
    worst = sorted(cos, key=cos.get)[:5]
    print(f"REPORT clip rn50 train step {dtype}: worst " + ", ".join(f"{k} cos {cos[k]:.5f} (fp32 gap {gap[k]:.1e})" for k in worst)
          + f"; median {sorted(cos.values())[len(cos) // 2]:.5f}; max fp32 gap {max(gap.values()):.1e}")
    head = {k: cos[k] for k in ("model.attnpool.q_proj.weight", "model.attnpool.k_proj.weight", "model.attnpool.v_proj.weight",
                                "model.attnpool.c_proj.linear.weight")}
    print(f"REPORT clip rn50 head {dtype}: " + ", ".join(f"{k.split('.')[-2]} {v:.5f}" for k, v in head.items()))
    assert min_cos is None or min(cos.values()) >= min_cos
    assert min(head.values()) >= head_cos and sorted(cos.values())[len(cos) // 2] >= median_cos
    new = plan.state_dict()
    rv = {k: _rel(new[k].cpu(), v) for k, v in ref["running_var"].items()}
    print(f"REPORT clip rn50 running_var {dtype}: max rel {max(rv.values()):.3e} ({max(rv, key=rv.get)})")
    assert max(rv.values()) < (1e-2 if dtype == "fp16" else 6e-2)      # measured: 6.0e-3 / 3.7e-2, both on the last block's bn3
    # the first AdamW step moves the weights by about lr; the packed operands follow the master weights
    k0 = "model.layer3.1.conv1.linear.weight"
    step = (new[k0].cpu() - sd[k0]).abs()
    assert 0.5e-4 < float(step.median()) < 1.5e-4
    lay = [l for l in plan.layers if l.name == "model.layer3.1.conv1"][0]
    o, c = sd[k0].shape[:2]
    packed = lay.fwd.b.float().cpu().view(o, -1)[:, :c]
    assert _rel(packed, new[k0].cpu().view(o, c)) < (1e-3 if dtype == "fp16" else 6e-3)
    kq = "model.attnpool.q_proj.weight"
    assert 0.5e-4 < float((new[kq].cpu() - sd[kq]).abs().median()) < 1.5e-4
    # the updated weights load into the inference plan, which embeds like the oracle with them (eval-mode BN: running_var)
    sd_new = {**sd_cal, **{k: v.cpu() for k, v in new.items()}}
    inf = CLIPResNetPlan(sd_new, nb, device="cuda", image_size=S, explain=False)
    emb = inf.embed(x6.cuda()).float().cpu()
    emb_ref = OR.OracleCLIPResNet(sd_new).forward(x6)
    print(f"REPORT clip rn50 {dtype}: embedding of the updated weights, rel err {_rel(emb, emb_ref):.2e}")
    assert _rel(emb, emb_ref) < 2e-2
    loss2 = float(plan.train_step(torch.from_numpy(imgs), _cos_loss(tg)))
    assert math.isfinite(loss2)


def test_captured_clip_train_step_equals_eager(bcosk_lib):
    """capture(): two graphs (forward; backward + optimizer + refresh) around the eager loss give the eager step's losses and weights,
    and capturing does not advance the training state."""
    S, nb, sd, imgs, tg = _rn50_case()
    imgs = torch.from_numpy(imgs)
    a = CLIPResNetTrainPlan(sd, nb, dtype="bf16", device="cuda", image_size=S)
    b = CLIPResNetTrainPlan(sd, nb, dtype="bf16", device="cuda", image_size=S)
    b.x_in.copy_(imgs)
    w0 = b.w_flat.clone()
    assert b.capture() and torch.equal(b.w_flat, w0) and float(b.adam_state[0]) == 0.0
    la, lb = [], []
    for _ in range(3):
        la.append(float(a.train_step(imgs, _cos_loss(tg))))
        lb.append(float(b.train_step(imgs, _cos_loss(tg))))
    torch.cuda.synchronize()
    assert float(b.adam_state[0]) == 3.0 and b.step_count == 3
    print(f"REPORT captured clip step: losses bit-identical {la == lb}, weights bit-identical {torch.equal(a.w_flat, b.w_flat)}")
    assert max(abs(x - y) / abs(x) for x, y in zip(la, lb)) < 1e-4, (la, lb)
    # split-K weight gradients add with fp32 atomics (order-dependent in the last bits), everything else is fixed-order
    assert _rel(b.w_flat, a.w_flat) < 1e-4


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs (NCCL all-reduce of the gradient buckets)")
def test_two_rank_clip_allreduce_matches_manual_sum():
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                          "--master-port", "29545", os.path.join(ROOT, "scripts", "exp_train_ddp.py"), "--arch", "clip_rn50"],
                         capture_output=True, text=True, timeout=900)
    line = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert line, out.stdout + out.stderr
    r = json.loads(line[-1])
    assert r["arch"] == "clip_rn50"
    assert r["grad_sum_rel_err_vs_manual_allreduce"] < 1e-5 and r["weights_identical_across_ranks"]
