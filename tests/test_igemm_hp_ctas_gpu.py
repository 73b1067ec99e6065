"""The three- and four-CTA-per-SM configurations of the parity-mode GEMM (include/bcosk.h `sched` = 3 / 4 with hp_accum,
csrc/bcosk_igemm_hp.cu hp::Cfg<64, 3> / <64, 4>) against the two-CTA one.

The two run the same MMAs in the same order and sum the partial accumulators with the same round-to-nearest fp32 adds in
the same order; only which warp does what, and when, differs.  So every output must be bit-identical: y planes, gains
(fp32 and 16-bit), mask bits and per-tile sums of squares.  Every output tensor is overwritten with a poison pattern before
each launch, so a launch that leaves part of a tensor unwritten cannot pass by leaving the other launch's bits in place.
"""
from __future__ import annotations

import math
import zlib

import pytest
import torch

import emulator as E
import opsutil as U
from bcos_b200 import _lib as L
from bcos_b200.engine import ops as O
from bcos_b200.engine.base import Act, PlanBase

OUT_FIELDS = ("y", "gain", "maskbits", "sq_out")
THREE_CTA_MAX_SMEM = (228 * 1024 - 3 * 1024) // 3        # shared memory per CTA with three CTAs on an SM
THREE_CTA_MAX_REGS = 96      # 18 warps put 5 on some SM sub-partitions: 5 warps x 96 x 32 registers <= 16 K per sub-partition
FOUR_CTA_MAX_SMEM = (228 * 1024 - 4 * 1024) // 4
FOUR_CTA_MAX_REGS = 80       # 24 warps: 6 per sub-partition, 6 x 80 x 32 <= 16 K


def ctas_fit(cfg, ctas_want=3) -> bool:
    """registers, spills, threads and shared memory of the three- (four-) CTA kernel admit three (four) CTAs per SM.  (The
    occupancy API reports 1 for every instance of this kernel, two-CTA ones included and at 0 bytes of shared memory, so it
    is recorded, not asserted: bcosk_igemm_hp_config in include/bcosk.h.)"""
    ctas, threads, smem, _, regs, local = cfg
    max_smem, max_regs = (THREE_CTA_MAX_SMEM, THREE_CTA_MAX_REGS) if ctas_want == 3 else (FOUR_CTA_MAX_SMEM, FOUR_CTA_MAX_REGS)
    return ctas == ctas_want and threads == 192 and smem <= max_smem and regs <= max_regs and local == 0


@pytest.fixture(scope="module")
def lib():
    from bcos_b200 import build
    build.build()
    return L.load()


@pytest.fixture
def hp_boxes(lib):
    """bcosk_set_hp_boxes for one test, restored afterwards"""
    prev = []

    def set_(v):
        prev.append(lib.bcosk_set_hp_boxes(v))

    yield set_
    for v in reversed(prev):
        lib.bcosk_set_hp_boxes(v)


def _gen(name):
    return torch.Generator().manual_seed(zlib.crc32(name.encode()))


def _act(g, nb, h, w, c, planes, dt):
    v = torch.randn(nb, h, w, c, generator=g)
    t = torch.zeros(nb, h, w, planes * c, dtype=dt)
    stored = E._split_store(t, v, planes)
    sq = (stored.double() ** 2).sum(-1).reshape(1, -1).float().contiguous()
    return Act(t, c, sq, 1)


def _conv_op(name, nb, h, cin, cout, k=1, stride=1, *, res=False, bn=False, chunk=0, dtype="fp16", gain32=False, kch=64):
    """one forward launch of the plane-aware kernel, built on the CPU and moved to the GPU"""
    g = _gen(name)
    dt = torch.float16 if dtype == "fp16" else torch.bfloat16
    plan = PlanBase(nb, planes=2, dtype=dtype, device="cpu", explain=True, explain_planes=2 if gain32 else 1)
    plan.flat_3x3 = False
    plan.hp_chunk = chunk
    x = _act(g, nb, h, h, cin, 2, dt)
    w = torch.randn(cout, cin, k, k, generator=g) / math.sqrt(cin * k * k)
    if bn:
        plan.sd = {"bn.running_var": torch.rand(cout, generator=g) + 0.5, "bn.weight": torch.rand(cout, generator=g) + 0.5}
        plan.fold_bn = False
    oh = (h + 2 * (k // 2) - k) // stride + 1
    r = _act(g, nb, oh, oh, cout, 2, dt) if res else None
    plan._conv_fwd("c", x, w, stride, k // 2, k // 2, bn="bn" if bn else None, relu=True, res=r, want_mask=True, kch=kch)
    op = plan.fwd_ops[-1]
    assert op.hp_accum and op.resolved_block_n() == 64 and op.mode == L.BCOSK_MODE_FWD
    assert (op.gain.dtype == torch.float32) == gain32
    memo = {}
    dops = [U.to_device(o, "cuda", memo) for o in plan.fwd_ops]
    for o in dops[:-1]:
        o.run()
    return dops[-1]


def _config(op, sched):
    op.sched = sched
    return L.igemm_hp_config(op.params())


def _run(op, sched, poison):
    op.sched = sched
    for f in OUT_FIELDS:
        t = getattr(op, f)
        if t is not None:
            t.view(torch.uint8).fill_(poison)
    op.run()
    torch.cuda.synchronize()
    return {f: getattr(op, f).clone() for f in OUT_FIELDS if getattr(op, f) is not None}


def check_identical(op, expect_three=True, expect_four=None) -> dict:
    """two-CTA (sched 1) vs three-CTA (sched 3) vs four-CTA (sched 4) launch of `op`: bit-identical outputs, each run twice.
    `expect_four`: whether sched 4 must run the four-CTA kernel (None: either, e.g. the launch has several drains)."""
    for f in ("res", "a"):
        t = getattr(op, f)
        assert t is None or t.data_ptr() != op.y.data_ptr(), (op.name, "y aliases an input")
    c2, c3, c4 = _config(op, 1), _config(op, 3), _config(op, 4)
    assert c2[0] == 2 and c2[5] == 0, c2
    if expect_three:
        assert ctas_fit(c3), c3
    if expect_four:
        assert ctas_fit(c4, 4), c4
    elif expect_four is False:
        assert c4 == c3, (c4, c3)
    runs = [(1, 0x5A), (3, 0xA5), (4, 0x96), (1, 0x3C), (3, 0xC3), (4, 0x69)]
    outs = [_run(op, s, poison) for s, poison in runs]
    for i in range(1, len(outs)):
        for f, ref in outs[0].items():
            got = outs[i][f]
            same = torch.equal(ref.view(torch.uint8), got.view(torch.uint8))
            if not same:
                diff = (ref.view(torch.uint8) != got.view(torch.uint8)).sum().item()
                raise AssertionError(f"{op.name}: {f} of run {i} (sched {runs[i][0]}) differs from sched 1 in {diff} bytes")
    return {"two": c2, "three": c3, "four": c4}


# ---- every 64-wide forward launch of ResNet-50 at a reduced batch -------------------------------------------------------------
@pytest.fixture(scope="module")
def rn50_plan(lib):
    from bcos_b200.models import synthetic_resnet_plan
    from bcos_b200.utils import synth
    plan = synthetic_resnet_plan("resnet50", 2, mode="parity", device="cuda", input_u8=True)
    plan.load_input(torch.from_numpy(synth.synth_images_u8(2, 224, 0)).cuda())
    plan.run_forward()
    torch.cuda.synchronize()
    return plan


def _rn50_launches(plan):
    return [op for op in plan.fwd_ops if isinstance(op, O.IgemmOp) and op.hp_accum and op.mode == L.BCOSK_MODE_FWD
            and op.resolved_block_n() == 64]


@pytest.mark.gpu
def test_rn50_launches_bit_identical(rn50_plan):
    ops = _rn50_launches(rn50_plan)
    assert len(ops) >= 30, len(ops)
    three = four = 0
    for op in ops:
        cfg = check_identical(op, expect_three=False)
        three += cfg["three"][0] == 3
        four += cfg["four"][0] == 4
        op.sched = 0
    print(f"\n{three} of {len(ops)} ResNet-50 64-wide forward launches run the three-CTA kernel with sched 3, {four} the four-CTA one with sched 4")
    assert four >= 6, four
    assert three >= len(ops) - 2, "the 64-wide ResNet-50 forward launches have the packed epilogue and fit the three-CTA kernel"


@pytest.mark.gpu
def test_three_ctas_resident(lib):
    """the new kernel's registers (no spills), threads and the shared-memory size the host picks admit three CTAs per SM"""
    for name, kw in [("occ_res_multi_drain", dict(cin=512, cout=128, res=True)), ("occ_res_one_drain", dict(cin=64, cout=256, res=True)),
                     ("occ_gain32", dict(cin=256, cout=64, res=True, gain32=True))]:
        op = _conv_op(name, 1, 14, kw.pop("cin"), kw.pop("cout"), **kw)
        c3, c4 = _config(op, 3), _config(op, 4)
        print("\n", name, "two-CTA", _config(op, 1), "three-CTA", c3, "sched 4", c4)
        assert ctas_fit(c3), c3
        if name == "occ_res_one_drain":
            assert ctas_fit(c4, 4), c4


# ---- K loops of 1 .. 16 paired stages, hp_chunk 1 / 2 / 4, with and without the residual, fp32 and 16-bit gains ----------
@pytest.mark.gpu
@pytest.mark.parametrize("gain32", [False, True], ids=["gain16", "gain32"])
@pytest.mark.parametrize("res", [False, True], ids=["plain", "res"])
@pytest.mark.parametrize("chunk", [1, 2, 4])
@pytest.mark.parametrize("stages", [1, 2, 4, 8, 16])
def test_k_loops_bit_identical(lib, stages, chunk, res, gain32):
    op = _conv_op(f"k{stages}_c{chunk}_{res}_{gain32}", 2, 12, 64 * stages, 128, res=res, bn=res, chunk=chunk, gain32=gain32)
    check_identical(op, expect_four=stages <= chunk and not gain32)


# ---- bf16 planes with chunked cross terms (unpaired stages), and M tails ------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [1, 2])
def test_bf16_chunked_cross_terms_bit_identical(lib, hp_boxes, chunk):
    hp_boxes(1 | 4)                 # no paired stages: every segment its own K loop, bf16 cross terms accumulated in chunks
    op = _conv_op(f"bf16_unpaired_{chunk}", 2, 10, 256, 64, res=True, chunk=chunk, dtype="bf16")
    check_identical(op)


@pytest.mark.gpu
def test_bf16_kch32_bit_identical(lib):
    """32-channel chunks (two chunks per K stage, never paired) with bf16 planes"""
    op = _conv_op("bf16_kch32", 2, 10, 32, 64, k=3, dtype="bf16", kch=32)
    check_identical(op)


@pytest.mark.gpu
@pytest.mark.parametrize("stages", [1, 4])
def test_m_tail_bit_identical(lib, stages):
    """M = 49: one partial tile (rows past M are computed and dropped)"""
    op = _conv_op(f"mtail_{stages}", 1, 7, 64 * stages, 64, res=True)
    assert op.M % 128 != 0
    check_identical(op)


@pytest.mark.gpu
def test_n_tail_declines(lib):
    """n = 72 (no packed epilogue): sched 3 falls back to the two-CTA kernel"""
    op = _conv_op("n72", 2, 9, 64, 72, k=3)
    assert _config(op, 3)[0] == 2
    check_identical(op, expect_three=False)
