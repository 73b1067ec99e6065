"""-m gpu: the DenseNet fine-tuning step (DenseNetTrainPlan, csrc/bcosk_dense_train.cu).

Kernel by kernel against the same arithmetic written with torch on the same 16-bit inputs; a small DenseNet (one block of three
layers, a transition, a one-layer block) against fp64 autograd with the same rounded weights, which isolates the concatenation
backward from the conditioning of a deep random-init network; then a whole DenseNet-121 step against the fp32 oracle.

Conditioning of the whole-step configuration (DenseNet-121, 64^2, batch 8, synthetic seed-0 weights, images seed 3): the
reference arithmetic's own gradients differ between fp32 and fp64 by a median of 1.5e-5 (relative, per tensor), the classifier's by
6.4e-6, every tensor but one by at most 1.9e-5, and norm0's BN weight by 2.2e-3 (its true gradient is ~0, see NORM0).  One 16-bit
plane (2^-11 fp16, 2^-8 bf16) is 4e3 / 3e4 times coarser than fp32; the per-tensor cosine floors below follow from that measured
sensitivity, as for the random-init ResNet-50 (tests/test_train_gpu.py).
"""
import json
import math
import os
import subprocess
import sys
import zlib

import pytest
import torch

import bcos_oracle as OR
from bcos_b200 import _lib as L
from bcos_b200.engine import DenseNetTrainPlan
from bcos_b200.engine import densenet as DN
from bcos_b200.utils import synth

pytestmark = pytest.mark.gpu
DT = {"bf16": torch.bfloat16, "fp16": torch.float16}
NBLK = 296
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# norm0's weight scales each channel of a block input; every consumer renormalises those channels with their batch statistics,
# so the loss does not depend on it (up to BN's eps): its true gradient is ~0 and what any finite precision computes is rounding
# noise (fp32 vs fp64: 2.2e-3 relative on DenseNet-121).  Its cosine is meaningless; it is only required to be finite.
NORM0 = "model.features.1.weight"


def _rel(a, b):
    return float((a.double() - b.double()).norm() / (b.double().norm() + 1e-300))


def _cos(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float(torch.dot(a, b) / (a.norm() * b.norm() + 1e-300))


def _gen(name):
    g = torch.Generator(device="cuda")
    g.manual_seed(zlib.crc32(name.encode()))
    return g


# prefixes 96 / 160 / 1024 at column 0 (consumers), a 32-wide slice at column 64 and a 96-wide one at column 40 (producers)
CASES = [(96, 0), (160, 0), (1024, 0), (32, 64), (96, 40)]


@pytest.mark.parametrize("c,col0", CASES)
@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
def test_slice_stats_and_consumer_finalize_match_torch(bcosk_lib, c, col0, dtype):
    rows = 1013                                     # not a multiple of the rows per block pass
    ld = col0 + c + 24
    dt, dtc = DT[dtype], L.DTYPE_CODE[dtype]
    g = _gen(f"stats{c}{col0}{dtype}")
    F = (torch.randn(rows, ld, device="cuda", generator=g) * 0.7 + 0.3).to(dt)
    part = torch.empty(NBLK, 2 * c, device="cuda")
    stats = [torch.full((ld,), -7.0, device="cuda") for _ in range(3)]
    L.dense_slice_stats(F, rows, ld, col0, c, 1e-5, part, *stats, dtc)
    x = F.double()[:, col0:col0 + c]
    var = x.var(0, unbiased=False)
    mean, v, rstd = (s[col0:col0 + c] for s in stats)
    assert _rel(mean, x.mean(0)) < 1e-6 and _rel(v, var) < 1e-5 and _rel(rstd, 1 / (var + 1e-5).sqrt()) < 1e-5
    outside = torch.cat([s[:col0] for s in stats] + [s[col0 + c:] for s in stats])
    assert bool((outside == -7.0).all())
    again = [torch.zeros(ld, device="cuda") for _ in range(3)]
    L.dense_slice_stats(F, rows, ld, col0, c, 1e-5, part, *again, dtc)
    assert all(torch.equal(a[col0:col0 + c], s[col0:col0 + c]) for a, s in zip(again, stats))
    # the consumer's alpha and running-variance EMA
    w = torch.rand(c, device="cuda", generator=g) + 0.5
    rv = torch.rand(c, device="cuda", generator=g) + 0.5
    rv0 = rv.clone()
    alpha = torch.empty(c, device="cuda")
    L.dense_consumer_finalize(v, rstd, w, c, 0.1, rv, alpha)
    torch.cuda.synchronize()
    assert _rel(alpha, w * rstd) < 1e-6 and _rel(rv, 0.9 * rv0 + 0.1 * v) < 1e-6


@pytest.mark.parametrize("c", [96, 160, 1024])
@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("gt_f32", [True, False])
def test_consumer_backward_matches_torch(bcosk_lib, c, dtype, gt_f32):
    """one pass: g_y = (g_t + t gnT) [t > 0], G[:, :c] += g_y alpha, S = sum g_y F; finalize: S rstd and K += -rstd^3 w S / M"""
    rows, ld = 1013, c + 64
    dt, dtc = DT[dtype], L.DTYPE_CODE[dtype]
    g = _gen(f"cons{c}{dtype}{gt_f32}")
    F = (torch.randn(rows, ld, device="cuda", generator=g) + 0.2).to(dt)
    alpha = torch.rand(c, device="cuda", generator=g) + 0.5
    t = (F.float()[:, :c] * alpha).clamp(min=0).to(dt)
    g_t = torch.randn(rows, c, device="cuda", generator=g) * 0.01
    g_t = g_t if gt_f32 else g_t.to(dt)
    gnt = torch.randn(rows, device="cuda", generator=g) * 0.01
    G0 = torch.randn(rows, ld, device="cuda", generator=g)
    K0 = torch.randn(ld, device="cuda", generator=g)
    rstd = torch.rand(c, device="cuda", generator=g) + 0.5
    w = torch.rand(c, device="cuda", generator=g) + 0.5
    gy = torch.where(t.float() > 0, g_t.float() + t.float() * gnt[:, None], torch.zeros((), device="cuda"))
    S = (gy.double() * F.double()[:, :c]).sum(0)
    for accumulate in (True, False):
        G, K = G0.clone(), K0.clone()
        part = torch.empty(NBLK, c, device="cuda")
        gw = torch.empty(c, device="cuda")
        L.dense_consumer_bwd(g_t, t, gnt, alpha, F, ld, rows, c, G, accumulate, part, dtc)
        L.dense_consumer_bwd_finalize(part, rstd, w, rows, c, accumulate, K, gw)
        torch.cuda.synchronize()
        want_G = (G0[:, :c] if accumulate else 0) + gy * alpha
        k = -(rstd.double() ** 3) * w * S / rows
        assert _rel(G[:, :c], want_G) < 1e-6 and torch.equal(G[:, c:], G0[:, c:])
        assert _rel(gw, S * rstd) < 1e-5
        assert _rel(K[:c], (K0[:c].double() if accumulate else 0) + k) < 1e-5 and torch.equal(K[c:], K0[c:])
        G2, K2, gw2 = G0.clone(), K0.clone(), torch.empty(c, device="cuda")
        L.dense_consumer_bwd(g_t, t, gnt, alpha, F, ld, rows, c, G2, accumulate, part, dtc)
        L.dense_consumer_bwd_finalize(part, rstd, w, rows, c, accumulate, K2, gw2)
        assert torch.equal(G2, G) and torch.equal(K2, K) and torch.equal(gw2, gw)


@pytest.mark.parametrize("c,col0", CASES)
@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
def test_slice_backward_matches_torch(bcosk_lib, c, col0, dtype):
    """g_out = G[:, slice] + (F[:, slice] - mean) K; producer conv: g_lin = 2 s g_out, gnT = -sum g_out F / n^2; block input: g_out"""
    rows, ld = 1013, col0 + c + 8
    dt, dtc = DT[dtype], L.DTYPE_CODE[dtype]
    g = _gen(f"slice{c}{col0}{dtype}")
    F = torch.randn(rows, ld, device="cuda", generator=g).to(dt)
    G = torch.randn(rows, ld, device="cuda", generator=g) * 0.01
    mean = torch.randn(ld, device="cuda", generator=g) * 0.1
    K = torch.randn(ld, device="cuda", generator=g) * 0.01
    s = (torch.rand(rows, c, device="cuda", generator=g) + 0.1).to(dt)
    inv_n = torch.rand(rows, device="cuda", generator=g) + 0.5
    sl = slice(col0, col0 + c)
    g_out = G[:, sl].double() + (F.double()[:, sl] - mean[sl].double()) * K[sl].double()
    out = torch.empty(rows, c, device="cuda", dtype=dt)
    gnt = torch.empty(rows, device="cuda")
    L.dense_slice_bwd(G, F, ld, col0, rows, c, mean, K, s, inv_n, out, gnt, dtc)
    torch.cuda.synchronize()
    tol = 4e-3 if dtype == "bf16" else 5e-4
    assert _rel(out.float(), 2 * g_out * s.double()) < tol
    assert _rel(gnt, -(g_out * F.double()[:, sl]).sum(1) * inv_n.double() ** 2) < 1e-5
    out2, gnt2 = torch.empty_like(out), torch.empty_like(gnt)
    L.dense_slice_bwd(G, F, ld, col0, rows, c, mean, K, s, inv_n, out2, gnt2, dtc)
    assert torch.equal(out2, out) and torch.equal(gnt2, gnt)
    L.dense_slice_bwd(G, F, ld, col0, rows, c, mean, K, None, None, out, None, dtc)
    torch.cuda.synchronize()
    assert _rel(out.float(), g_out) < tol


def _small_arch(monkeypatch):
    arch = "densenet_3l_t"
    cfg = (64, (3, 1), 64)         # one block of three layers (growth 64: the transition's 128 outputs suit the ResNet train kernels),
                                   # a transition, a one-layer block
    monkeypatch.setitem(DN.DENSENET_ARCH, arch, cfg)
    monkeypatch.setitem(OR.DENSENET_ARCH, arch, cfg)
    return arch


def test_small_densenet_step_matches_fp64_autograd(bcosk_lib, monkeypatch):
    """Three dense layers and a transition in train mode against fp64 autograd with the SAME 16-bit-rounded conv weights: every
    conv weight gradient, every BN weight gradient (the consumers' norm1 / transition norm / norm5 and the norm2s), the running
    variances and the loss.  The gradient wrt the block input reaches the weights only through the stem, so the stem's weight and
    norm0 gradients check it."""
    arch = _small_arch(monkeypatch)
    S, nb = 64, 4
    sd = synth.synth_state_dict(OR.densenet_state_shapes(arch), 0)
    imgs = synth.synth_images_u8(nb, S, 5)
    labels = torch.arange(nb) * 71 % 1000
    sd16 = {k: (v.to(torch.float16).float() if k.endswith(".linear.weight") else v) for k, v in sd.items()}
    sd64 = {k: (v.double() if v.is_floating_point() else v) for k, v in sd16.items()}
    x64 = synth.to_bcos_input(imgs).double()
    om = OR.OracleDenseNet(arch, sd64)
    om.calibrate_bn(x64)
    ref = OR.train_step_reference(om, x64, labels)
    sd_plan = {k: (v.float() if v.is_floating_point() else v) for k, v in sd64.items()}      # calibrated running variances
    plan = DenseNetTrainPlan(arch, sd_plan, nb, dtype="fp16", device="cuda", image_size=S, loss_scale=65536.0)
    loss = plan.train_step(torch.from_numpy(imgs), labels)
    torch.cuda.synchronize()
    assert abs(float(loss) - float(ref["loss"])) <= 2e-4 * float(ref["loss"])
    g = plan.gradients()
    assert set(g) == set(ref["grads"])
    assert math.isfinite(float(g[NORM0].abs().sum()))
    cos = {k: _cos(g[k].cpu(), r) for k, r in ref["grads"].items() if k != NORM0}
    rel = {k: _rel(g[k].cpu(), r) for k, r in ref["grads"].items() if k != NORM0}
    worst = min(cos, key=cos.get)
    print(f"REPORT small densenet fp16: min cos {cos[worst]:.6f} ({worst}) max rel {max(rel.values()):.3e} ({max(rel, key=rel.get)})")
    assert cos[worst] >= 0.9995 and max(rel.values()) < 0.03
    new = plan.state_dict()
    for k, v in ref["running_var"].items():
        assert _rel(new[k].cpu(), v) < 2e-3, k


def _densenet121_case():
    arch, S, nb = "densenet121", 64, 8
    sd = synth.synth_state_dict(OR.densenet_state_shapes(arch), 0)
    imgs = synth.synth_images_u8(nb, S, 3)
    labels = torch.arange(nb) * 41 % 1000
    return arch, S, nb, sd, imgs, labels


@pytest.mark.parametrize("dtype,loss_scale,min_cos", [("fp16", 65536.0, 0.995), ("bf16", 1.0, 0.92)])
def test_densenet121_train_step_matches_oracle(bcosk_lib, dtype, loss_scale, min_cos):
    """`min_cos` holds for every tensor whose fp32 gradient is within 1e-4 of fp64: all but norm0's weight (see NORM0), which only
    has to stay finite.  The others are 1.4e-5 .. 1.9e-5 from fp64 in fp32; measured on a B200 they reach cosines of 0.9978
    (fp16) and 0.945 (bf16), i.e. the 16-bit rounding of one plane amplified as the fp32 gap predicts."""
    arch, S, nb, sd, imgs, labels = _densenet121_case()
    sd64 = {k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}
    om = OR.OracleDenseNet(arch, sd)
    om.calibrate_bn(synth.to_bcos_input(imgs))
    ref = OR.train_step_reference(om, synth.to_bcos_input(imgs), labels)
    om64 = OR.OracleDenseNet(arch, sd64)
    om64.calibrate_bn(synth.to_bcos_input(imgs).double())
    ref64 = OR.train_step_reference(om64, synth.to_bcos_input(imgs).double(), labels)
    gap = {k: _rel(r, ref64["grads"][k]) for k, r in ref["grads"].items()}
    plan = DenseNetTrainPlan(arch, sd, nb, dtype=dtype, device="cuda", image_size=S, loss_scale=loss_scale)
    loss = plan.train_step(torch.from_numpy(imgs), labels)
    torch.cuda.synchronize()
    assert abs(float(loss) - float(ref["loss"])) <= 1e-3 * float(ref["loss"])
    g = plan.gradients()
    assert set(g) == set(ref["grads"])
    cos = {k: _cos(g[k].cpu(), r) for k, r in ref["grads"].items()}
    fc = cos["model.classifier.linear.weight"]
    well = {k: c for k, c in cos.items() if gap[k] < 1e-4}
    worst = sorted(cos, key=cos.get)[:5]
    print(f"REPORT densenet121 train step {dtype}: worst " + ", ".join(f"{k} cos {cos[k]:.5f} (fp32 gap {gap[k]:.1e})" for k in worst)
          + f"; median {sorted(cos.values())[len(cos) // 2]:.5f} fc {fc:.6f}; {len(well)} of {len(cos)} tensors with gap < 1e-4")
    assert set(cos) - set(well) <= {NORM0} and all(math.isfinite(float(v.abs().sum())) for v in g.values())
    assert min(well.values()) >= min_cos and fc >= (0.9999 if dtype == "fp16" else 0.995)
    # every consumer's running_var follows its own EMA of the batch variance of the channels it reads
    new = plan.state_dict()
    rv_rel = {k: _rel(new[k].cpu(), v) for k, v in ref["running_var"].items()}
    print(f"REPORT densenet121 running_var {dtype}: max rel {max(rv_rel.values()):.3e} ({max(rv_rel, key=rv_rel.get)})")
    assert max(rv_rel.values()) < (2e-3 if dtype == "fp16" else 3e-2)
    # the first AdamW step moves the weights by about lr; the packed operands follow the master weights
    k0 = "model.features.6.denselayer3.conv1.linear.weight"
    step = (new[k0].cpu() - sd[k0]).abs()
    assert 0.5e-4 < float(step.median()) < 1.5e-4
    lay = [l for l in plan.layers if l.name == "model.features.6.denselayer3.conv1"][0]
    o, c = sd[k0].shape[:2]
    packed = lay.fwd.b.float().cpu().view(o, -1)[:, :c]
    assert _rel(packed, new[k0].cpu().view(o, c)) < (1e-3 if dtype == "fp16" else 6e-3)
    loss2 = float(plan.train_step(torch.from_numpy(imgs), labels))
    assert math.isfinite(loss2)


def test_captured_densenet_train_step_equals_eager(bcosk_lib):
    """DenseNetTrainPlan.capture(): the whole step as one CUDA graph gives the eager step's losses and weights; capturing does
    not advance the training state."""
    arch, S, nb, sd, imgs, labels = _densenet121_case()
    imgs = torch.from_numpy(imgs)
    a = DenseNetTrainPlan(arch, sd, nb, dtype="bf16", device="cuda", image_size=S)
    b = DenseNetTrainPlan(arch, sd, nb, dtype="bf16", device="cuda", image_size=S)
    b.load_batch(imgs, labels)
    w0 = b.w_flat.clone()
    assert b.capture() and torch.equal(b.w_flat, w0) and float(b.adam_state[0]) == 0.0
    la, lb = [], []
    for _ in range(3):
        la.append(float(a.train_step(imgs, labels)))
        lb.append(float(b.train_step(imgs, labels)))
    torch.cuda.synchronize()
    assert float(b.adam_state[0]) == 3.0 and b.step_count == 3
    assert max(abs(x - y) / abs(x) for x, y in zip(la, lb)) < 1e-4, (la, lb)
    # split-K weight gradients add with fp32 atomics (order-dependent in the last bits), everything else is fixed-order
    assert _rel(b.w_flat, a.w_flat) < 1e-4


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs (NCCL all-reduce of the gradient buckets)")
def test_two_rank_densenet_allreduce_matches_manual_sum():
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                          "--master-port", "29543", os.path.join(ROOT, "scripts", "exp_train_ddp.py"), "--arch", "densenet121"],
                         capture_output=True, text=True, timeout=900)
    line = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert line, out.stdout + out.stderr
    r = json.loads(line[-1])
    assert r["arch"] == "densenet121"
    assert r["grad_sum_rel_err_vs_manual_allreduce"] < 1e-5 and r["weights_identical_across_ranks"]
