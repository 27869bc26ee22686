"""Runs only the roofline probe of bench.py (back-to-back steady fused sub-step launches on job-shaped
operands) so that `ncu --set full -k regex:substep_kernel` can capture a few of them cheaply.

    ncu --set full --clock-control none --import-source on -k regex:substep_kernel -s 170 -c 3 \
        -o gpurun_out/prof python profiles/burst_probe.py --requests 128
"""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from lanpaint_b200.engine import LanPaint, pack_mask  # noqa: E402
from lanpaint_b200.runner import SynthDenoiser, VESampling, time_steady_substep  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--requests", type=int, default=128)
ap.add_argument("--rng", default="philox")
ap.add_argument("--no-merge", action="store_true")
ap.add_argument("--mask", default="random", choices=["random", "blob"])
ap.add_argument("--tma", type=int, default=1, help="0 = LDG, 1 = TMA-staged (default)")
ap.add_argument("--rotate", type=int, default=3, help="independent operand sets cycled (1 = L2-assisted)")
args = ap.parse_args()
dev = torch.device("cuda:0")
from lanpaint_b200 import _native  # noqa: E402
_native.load().lp_set_option(b"tma", args.tma)
shape = (args.requests, 4, 128, 128)
g = torch.Generator().manual_seed(0)
y = torch.randn(shape, generator=g).to(dev)
if args.mask == "blob":
    mask = torch.ones((args.requests, 1, 128, 128))
    mask[:, :, 19:109, 19:109] = 0.0
    mask = mask.to(dev)
else:
    mask = (torch.rand((args.requests, 1, 128, 128), generator=g) < 0.5).float().to(dev)
eng = LanPaint(SynthDenoiser(VESampling()), 5, 15.0, 5.0, 1.0, 0.2, MinStepFrac=1.0, rng=args.rng,
               merge_noise=not args.no_merge)
ts = time_steady_substep(eng, y, pack_mask(mask, y), sigma=2.0, launches=53, repeats=5, rotate=args.rotate)
print("per-launch us:", [round(t, 2) for t in ts])
