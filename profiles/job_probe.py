"""runner.GraphedJob (whole-job graph, device-resident inputs) at a given batch size: ms per job.

    python profiles/job_probe.py --requests 256 [--rng philox] [--net two_head|cond_uncond]
The library's LANPAINT_B200_TMA environment switch applies."""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from lanpaint_b200.engine import CfgPair, LanPaint, pack_mask  # noqa: E402
from lanpaint_b200.runner import GraphedJob, HostSchedule, SynthCondNet, SynthDenoiser, VESampling, karras_sigmas  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--requests", type=int, default=128)
ap.add_argument("--rng", default="philox")
ap.add_argument("--net", default="two_head", choices=["two_head", "cond_uncond"])
ap.add_argument("--jobs", type=int, default=20)
args = ap.parse_args()
dev = torch.device("cuda:0")
R = args.requests
shape = (R, 4, 128, 128)


class Guider:
    def __init__(self):
        self.inner_model, self.model_sampling, self.net = self, VESampling(), SynthCondNet()

    def __call__(self, x, t, model_options=None, seed=None):
        return CfgPair(self.net(x, t, 0.3), self.net(x, t, -0.2), 5.0, 5.0)


model = SynthDenoiser(VESampling()) if args.net == "two_head" else Guider()
eng = LanPaint(model, NSteps=5, Friction=15.0, Lambda=5.0, Beta=1.0, StepSize=0.2, MinStepFrac=1.0, rng=args.rng,
               batched_replace="per_sample")
sched = HostSchedule(karras_sigmas(20), R, 5)
g = torch.Generator().manual_seed(0)
y, noise = torch.randn(shape, generator=g).to(dev), torch.randn(shape, generator=g).to(dev)
pm = pack_mask((torch.rand((R, 1, 128, 128), generator=g) < 0.5).to(dev), y)
job = GraphedJob(eng, sched, shape, dev)
for _ in range(3):
    job.run(y, noise, pm)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(args.jobs):
    job.run(y, noise, pm)
e1.record()
torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / args.jobs
print(f"R={R} rng={args.rng} net={args.net}: {ms:.3f} ms per job, {R * sched.substeps / ms * 1e3:.0f} sub-steps/s, "
      f"{job.launches + job.model_calls} graph nodes")
