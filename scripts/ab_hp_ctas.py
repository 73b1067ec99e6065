"""Two vs three vs four CTAs per SM on the 64-wide parity-mode forward launches (include/bcosk.h `sched` with hp_accum): time every
such launch of the ResNet-50 plan (batch 256, 224^2, `parity` mode) under each configuration, alternating them, with CUDA events
around warmed launches.  Prints one line per launch (ms, GB/s over IgemmOp.algo_bytes(), the configuration autotune keeps) and a
JSON summary with the GPU name and power limit read in the same run.

  python scripts/ab_hp_ctas.py [--batch 256 --reps 20 --rounds 3 --json OUT.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from bcos_b200 import _lib as L  # noqa: E402
from bcos_b200 import build as bbuild  # noqa: E402
from bcos_b200.engine import ops as O  # noqa: E402
from bcos_b200.models import synthetic_resnet_plan  # noqa: E402
from bcos_b200.utils import synth  # noqa: E402


def gpu_info(dev: int) -> dict:
    info = {"gpu": torch.cuda.get_device_name(dev)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info.update(power_limit_w=float(q[0]), max_sm_clock_mhz=float(q[1]))
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        info.update(power_limit_w=None, max_sm_clock_mhz=None)
    return info


def time_op(op, reps: int) -> float:
    """median ms of `reps` launches, each between two events, after two warm-up launches"""
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    op.run()
    op.run()
    ts = []
    for _ in range(reps):
        ev[0].record()
        op.run()
        ev[1].record()
        ev[1].synchronize()
        ts.append(ev[0].elapsed_time(ev[1]))
    return sorted(ts)[len(ts) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--arch", default="resnet50")
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the two configurations per launch (min over rounds)")
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    bbuild.build()
    L.require_device()
    dev = torch.cuda.current_device()
    plan = synthetic_resnet_plan(args.arch, args.batch, mode="parity", device="cuda", input_u8=True)
    imgs = torch.from_numpy(synth.synth_images_u8(min(args.batch, 64), 224, 1000))
    plan.load_input(imgs.repeat((args.batch + imgs.shape[0] - 1) // imgs.shape[0], 1, 1, 1)[:args.batch].contiguous().cuda())
    plan.run_forward()
    torch.cuda.synchronize()
    ops = [op for op in plan.fwd_ops if isinstance(op, O.IgemmOp) and op.hp_accum and op.mode == L.BCOSK_MODE_FWD
           and op.resolved_block_n() == 64]
    info = gpu_info(dev)
    print(f"# {info['gpu']}, power limit {info['power_limit_w']} W, max SM clock {info['max_sm_clock_mhz']} MHz; "
          f"{args.arch} batch {args.batch}, parity mode, {len(ops)} 64-wide forward launches")
    print(f"{'launch':32s} {'K':>5s} {'N':>5s} {'CTAs':>4s} {'ms 2-CTA':>9s} {'ms 3-CTA':>9s} {'ms s4':>9s} {'GB/s 2':>7s} {'GB/s best':>9s} "
          f"{'gain':>6s} keep")
    rows = []
    for op in ops:
        op.sched = 3
        ctas3 = L.igemm_hp_config(op.params())[0]
        op.sched = 4
        ctas4 = L.igemm_hp_config(op.params())[0]
        t = {1: [], 3: [], 4: []}
        for _ in range(args.rounds):
            for s in t:
                op.sched = s
                t[s].append(time_op(op, args.reps))
        ms = {s: min(v) for s, v in t.items()}
        keep = 1
        for s in (3, 4):                                  # the tie rule of PlanBase.autotune
            if ms[s] < ms[keep] * 0.98:
                keep = s
        op.sched = 0
        gb = op.algo_bytes() / 1e9
        row = {"name": op.name, "K": op.ktot, "N": op.n, "M": op.M, "ctas_sched3": ctas3, "ctas_sched4": ctas4, "ms_two": ms[1],
               "ms_three": ms[3], "ms_sched4": ms[4], "ms_kept": ms[keep], "gbs_two": gb / (ms[1] * 1e-3), "gbs_kept": gb / (ms[keep] * 1e-3),
               "keep_sched": keep}
        rows.append(row)
        print(f"{op.name:32s} {op.ktot:5d} {op.n:5d} {ctas4:4d} {ms[1]:9.4f} {ms[3]:9.4f} {ms[4]:9.4f} {row['gbs_two']:7.0f} "
              f"{row['gbs_kept']:9.0f} {(ms[1] - ms[keep]) / ms[1] * 100:5.1f}% {keep}")
    s1 = sum(r["ms_two"] for r in rows)
    sb = sum(r["ms_kept"] for r in rows)
    summary = {**info, "arch": args.arch, "batch": args.batch, "launches": len(rows), "ms_two_total": s1, "ms_autotuned_total": sb,
               "moved": sum(r["keep_sched"] != 1 for r in rows), "rows": rows}
    print(f"# sum over these launches: two CTAs {s1:.3f} ms, per-launch choice {sb:.3f} ms ({summary['moved']} launches moved)")
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as fh:
            json.dump(summary, fh, indent=1)


if __name__ == "__main__":
    main()
