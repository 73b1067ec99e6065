"""Workload for ncu: 2 warm eager steps of the RN50 plan, then either one full step or a few selected launches.

  ncu --metrics gpu__time_duration.sum --clock-control none -s 334 -c 167 --csv --log-file gpurun_out/launches.csv \
      python scripts/profile_step.py
  ncu --set full --clock-control none --import-source on -k regex:bcosk_igemm -s 214 -c 4 -o gpurun_out/prof \
      python scripts/profile_step.py --only model.layer1.1.conv3,model.layer3.1.conv2,model.layer1.1.conv1.dgrad,model.layer3.1.conv2.dgrad
"""
import argparse, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from bcos_b200.models import synthetic_resnet_plan
from bcos_b200.utils import synth

ap = argparse.ArgumentParser()
ap.add_argument("--batch", type=int, default=256)
ap.add_argument("--arch", default="resnet50")
ap.add_argument("--only", default="")
ap.add_argument("--mode", default=None, help="engine/resnet.py PRECISION_MODES name (default: parity); overrides --planes / --dtype")
ap.add_argument("--planes", type=int, default=None)
ap.add_argument("--dtype", default=None, choices=["bf16", "fp16"])
ap.add_argument("--autotune", type=int, default=0, help="pick per-launch schedules first (as capture() does); use with ncu --profile-from-start off")
a = ap.parse_args()
if a.planes is None and a.dtype is None:
    plan = synthetic_resnet_plan(a.arch, a.batch, mode=a.mode or "parity", device="cuda", input_u8=True)
else:
    plan = synthetic_resnet_plan(a.arch, a.batch, planes=a.planes or 1, dtype=a.dtype or "bf16", device="cuda", input_u8=True,
                                seed_scale=4096.0 if a.dtype == "fp16" else 1.0)
imgs = torch.from_numpy(synth.synth_images_u8(32, 224, 5)).repeat((a.batch + 31) // 32, 1, 1, 1)[:a.batch].contiguous()
plan.load_input(imgs)
ops = plan.fwd_ops + plan.bwd_ops
sel = [s for s in a.only.split(",") if s]
if a.autotune:
    plan.autotune()
for _ in range(1 if sel else 2):
    for o in ops:
        o.run()
torch.cuda.synchronize()
n_tile = sum(1 for o in ops if type(o).__name__ == "IgemmOp" and not o.flat)
print("per-tile/persistent igemm launches in the warm step:", n_tile, "(use as ncu --launch-skip with -k regex:bcosk_igemm)")
torch.cuda.profiler.start()          # ncu --profile-from-start off captures only this step
for o in ops:
    if not sel or o.name in sel:
        o.run()
torch.cuda.synchronize()
torch.cuda.profiler.stop()
print("launches per step", len(ops), "igemm", sum(type(o).__name__ == "IgemmOp" for o in ops))
