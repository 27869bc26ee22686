#!/usr/bin/env python
"""bench.py -- Langevin sub-steps/sec on the SDXL 128x128x4 latent (BASELINE.json's metric).

    python bench.py --gpus N --steps K --warmup W              # this repo (CUDA kernels), through the node API
    python bench.py --impl reference --gpus N --steps K ...    # the reference's CPU path on the host cores
    python bench.py ... --dump-outputs DIR                     # also write what the last timed step returned (.npy)

What is measured (`config.workload`): `requests_per_gpu` independent SDXL inpaint requests of shape [1,4,128,128]
(BASELINE configs[1]'s latent) batched per GPU, each running the reference schedule: karras-20 sigmas x N=5 think
steps with the node defaults (MinStepFrac=1, EarlyStop=1) = 53 Langevin sub-steps + 20 final denoises = 73 guider
evaluations (146 network calls: cond + uncond) per request (SURVEY 8d), a pointwise synthetic network standing in
for the UNet, sampler "euler".

Every job goes through the reference-facing plugin call: `comfy_nodes.LanPaint_KSampler.sample(model, seed, steps,
cfg, "euler", "karras", positive, negative, LATENT, ...)` -- ComfyUI replaced by `minicomfy` -- with a LATENT dict of
pinned HOST tensors in and a LATENT dict of host tensors out.  One bench "step" = `jobs_per_step` such calls.
  value   request-sub-steps/s over the DEVICE time of the sampler loop inside those calls (two CUDA events recorded
          by the node layer once the inputs are on the device / after the last kernel; max over ranks of the sum)
  e2e     the same calls by the wall clock: ComfyUI's CPU-side prepare_noise, H2D of latent / noise / mask, the
          sampler loop, D2H of the result
The line is emitted for the shipped default rng="torch" (the reference's own randn stream: same seed, same latent);
`variants.philox` holds the same measurement for the cheaper counter-based stream, `serving` the host-owned
`runner.GraphedJob` numbers (round-1's headline path), `configs` the literal BASELINE configurations.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

SHAPE = (4, 128, 128)          # SDXL latent of a 1024x1024 image
N_OUTER, N_INNER = 20, 5
METRIC = "Langevin sub-steps/sec (SDXL 128x128x4 latent, N=5)"


def algo_bytes_per_elem(channels: int, head_bytes: int = 4) -> float:
    """SURVEY 8d: read x, y, C (fp32) + two heads + write x, C (fp32) + uint8 spatial mask."""
    return 12.0 + 2.0 * head_bytes + 8.0 + 1.0 / channels


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------
# clocks: NVML sampled in-process from before the warm-up until after the timed region
# ------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index: int, period: float = 0.02):
        self.index, self.period = index, period
        self.rows, self.marks, self.stop_flag, self.thread, self.err = [], {}, False, None, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()
        except Exception as e:  # no NVML: the line says so instead of inventing numbers
            self.err = f"{type(e).__name__}: {e}"
        return self

    def _loop(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    rs = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    rs = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.rows.append((time.perf_counter(), sm, rs))
            except Exception as e:
                self.err = f"{type(e).__name__}: {e}"
            time.sleep(self.period)

    def mark(self, name):
        self.marks[name] = time.perf_counter()

    def stop(self):
        self.stop_flag = True
        if self.thread is not None:
            self.thread.join(timeout=1.0)

    def summary(self):
        t0, t1 = self.marks.get("t0", 0.0), self.marks.get("t1", float("inf"))
        inside = [(sm, rs) for (t, sm, rs) in self.rows if t0 <= t <= t1]
        sm = sorted(v for v, _ in inside)
        reasons = set()
        for _, rs in inside:
            for bit, name in self.REASONS.items():
                if rs & bit:
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_min_mhz": sm[0] if sm else None,
                "sm_max_mhz": getattr(self, "max_sm", None), "reasons": sorted(reasons),
                "samples": len(sm), "samples_total": len(self.rows), "source": "NVML in-process, 20 ms period, "
                "samples inside the timed region", "error": self.err}


def bind_to_gpu_numa_node(index: int):
    """Best effort: run this rank (and first-touch its pinned buffers) on the NUMA node its GPU hangs off, so
    eight ranks do not push their H2D/D2H traffic through one socket.  Returns the node or None."""
    try:
        p = torch.cuda.get_device_properties(index)
        bdf = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if allowed:
            os.sched_setaffinity(0, allowed)
            return node
    except Exception:
        pass
    return None


def dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


# ------------------------------------------------------------------------------------------
# the reference arm: the reference's own engine (oracle/_ref, bytecode compiled from /root/reference) when it was
# built, else the oracle port (op-for-op restatement), on the host cores.  The one place outside tests/ where
# oracle/ is executed.
# ------------------------------------------------------------------------------------------
def reference_engine_kind():
    from oracle import build_ref
    return "reference" if build_ref.load() is not None else "port"


def reference_nodes():
    """The reference's own node module (oracle/_ref bytecode of nodes.py, imported over minicomfy) or None."""
    from oracle import build_ref
    return build_ref.load_nodes()


REFERENCE_API = ("the reference's own LanPaint_KSampler.sample (oracle/_ref bytecode of nodes.py + lanpaint.py, ComfyUI "
                 "replaced by minicomfy as in the GPU arm), LATENT dict in -> LATENT dict out")


def cpu_node_job(ref_nodes, requests: int, threads: int, seed: int = 0):
    """ONE call of the UNMODIFIED reference's `LanPaint_KSampler.sample` on `requests` requests on the host cores:
    the very call the GPU arm times (same arguments, same conditioning, euler / karras-20 / N=5, the synthetic
    network as its torch formula), through the reference's own patched CFGGuider / KSAMPLER / per-sigma wrapper
    (nodes.py:161-216, 229-379, 487-513) into `LanPaint.__call__`.  ComfyUI's CPU prepare_noise and the LATENT
    dict hand-over are inside the timed region, as they are in the GPU arm's e2e.
    Returns (seconds, request-sub-steps done)."""
    import contextlib
    import io
    import minicomfy
    torch.set_num_threads(threads)
    g = torch.Generator().manual_seed(seed)
    y = torch.randn((requests,) + SHAPE, generator=g)
    nm = (torch.rand((requests, 1) + SHAPE[1:], generator=g) < 0.5).float()
    calls = [0]

    def net(x, sigma, cond):        # lanpaint_b200.runner.SynthCondNet's formula (lp_synth_denoiser_f32)
        calls[0] += 1
        return 0.7 * x + 0.1 * torch.tanh(x) + float(cond)

    patcher = minicomfy.ModelPatcher(minicomfy.BaseModel(net), "cpu")
    node = ref_nodes.NODE_CLASS_MAPPINGS["LanPaint_KSampler"]()
    t0 = time.perf_counter()
    with contextlib.redirect_stdout(io.StringIO()):      # the reference prints from outer_sample (nodes.py:179)
        (out,) = node.sample(patcher, 1000 + seed, N_OUTER, 5.0, "euler", "karras", 0.3, -0.2,
                             {"samples": y, "noise_mask": nm}, 1.0, N_INNER, "Image First", "", "🖼️ Image Inpainting")
    dt = time.perf_counter() - t0
    assert calls[0] == 2 * 73 and out["samples"].shape == y.shape, (calls[0], out["samples"].shape)
    return dt, requests * 53


def calibrate_threads(requests: int) -> int:
    """The reference's eager path is ~90 small element-wise ops per sub-step; on a many-core host more
    threads can be much slower (fork/join per op).  Time ONE outer step of the actual workload (5 sub-steps,
    6 model calls) per candidate thread count and keep the fastest, so the CPU arm is the best this host can
    do rather than a strawman."""
    cores = os.cpu_count() or 1
    best, best_t = 1, float("inf")
    for c in sorted({k for k in (2, 4, 8, 16, 32, 64, cores) if k <= cores}):
        warm = cpu_job(requests, 1, c)[0]      # also warms this thread count
        if warm > 2.5 * best_t:                # past the knee: more threads only get slower on this host
            break
        dt = min(cpu_job(requests, 1, c)[0] for _ in range(2))
        if dt < best_t:
            best, best_t = c, dt
    return best


def cpu_job(requests: int, outer_steps: int, threads: int, seed: int = 0):
    """Runs the first `outer_steps` outer steps of the workload on `requests` requests on the CPU: k-diffusion's
    Euler loop and the per-sigma schedule glue (oracle restatement of nodes.py:229-315) around the engine -- the
    reference's own `LanPaint.__call__` when oracle/_ref is built, the port's `outer_step` otherwise.
    Returns (seconds, request-sub-steps done)."""
    from oracle import build_ref
    from oracle import langevin_oracle as O
    torch.set_num_threads(threads)
    g = torch.Generator().manual_seed(seed)
    shape = (requests,) + SHAPE
    y, noise = torch.randn(shape, generator=g), torch.randn(shape, generator=g)
    dm = (torch.rand((requests, 1) + SHAPE[1:], generator=g) < 0.5).float().expand(shape).contiguous()
    sig = O.karras_sigmas(N_OUTER)
    hp = O.Hyper(n_steps=N_INNER, min_step_frac=1.0)
    model = O.PointwiseDenoiser(O.VESampling())
    Ref = build_ref.load()
    ref_engine = None
    if Ref is not None:
        ref_engine = Ref(model, N_INNER, 15.0, hp.lam, hp.beta, hp.step_size, IS_FLUX=False, IS_FLOW=False, MinStepFrac=1.0)
    t0 = time.perf_counter()
    x = model.model_sampling.noise_scaling(sig[0], noise, y)
    mask = O.binarise_mask(dm)
    s_in = x.new_ones([x.shape[0]])
    sub = 0
    for i in range(min(outer_steps, N_OUTER)):
        sigma = sig[i] * s_in
        tm = O.times_from_sigma(sigma, False)
        n_eff = O.inner_steps_for(sigma, sig, tm.abt, hp.n_steps, 1, 1.0)   # position in the FULL schedule
        if ref_engine is not None:
            den = ref_engine(x, y, noise, sigma, mask, tuple(tm), {}, 0, n_steps=n_eff)   # rewrites x in place
        else:
            den, x = O.outer_step(model, x, y, noise, sigma, mask, tm, hp, n_eff)
        x = x + (x - den) / sigma.view(-1, 1, 1, 1) * (sig[i + 1] - sig[i])
        sub += n_eff
    return time.perf_counter() - t0, sub * requests


def run_reference(args):
    import warnings
    warnings.filterwarnings("ignore")   # the reference's autocast(float32) wrappers warn on CPU (lanpaint.py:201,239)
    rank, world, _ = dist_env()
    if rank != 0:
        return
    host_cores = os.cpu_count() or 1
    req = args.ref_requests
    kind = reference_engine_kind()
    ref_nodes = reference_nodes() if kind == "reference" else None
    cores = calibrate_threads(req)

    def job(seed):
        if ref_nodes is not None:
            return cpu_node_job(ref_nodes, req, cores, seed)
        return cpu_job(req, N_OUTER, cores, seed)

    for k in range(args.warmup):
        job(k)
    t, units = 0.0, 0
    for k in range(args.steps):
        dt, u = job(100 + k)
        t += dt
        units += u
    value = units / t
    sample = (f"{req} requests per step (the GPU arm batches {args.requests} per call), full karras-20 x N=5 schedule "
              f"(53 sub-steps/request); {cores} torch threads (fastest of a probe over 1..{host_cores} host cores); "
              + (REFERENCE_API if ref_nodes is not None else
                 "engine = the reference's own LanPaint.__call__ (oracle/_ref bytecode) under the oracle's Euler loop"
                 if kind == "reference" else "oracle port"))
    cfg = workload_config(args, "reference")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "sub-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / max(1, args.steps),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": value, "unit": "sub-steps/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "sub-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if ref_nodes is not None:
        line["config"]["api"] = REFERENCE_API
        line["e2e"]["api"] = REFERENCE_API
    print(json.dumps(line), flush=True)


def workload_config(args, impl="b200"):
    n_el = args.requests * SHAPE[0] * SHAPE[1] * SHAPE[2]
    touched = 5.25 * 4 * n_el / 1e6
    cfg = {"workload": "sdxl_1024_inpaint_4x128x128_karras20_N5", "requests_per_gpu": args.requests,
           "latent_shape": [1] + list(SHAPE), "outer_steps": N_OUTER, "think_steps": N_INNER,
           "substeps_per_request": 53, "model_calls_per_request": 73,
           "reference_requests": args.ref_requests,
           "reference_requests_note": "the CPU arm runs a bounded sample of this many requests per step; CPU per-request "
                                      "throughput rises with batch (BASELINE.md 3), so the CPU figure is a lower bound "
                                      "of what a larger CPU batch would reach (up to ~2x)",
           "denoiser": "synthetic pointwise network (one kernel per cond / uncond evaluation)", "sampler": "euler",
           "mask": "random 50% per spatial site" if args.mask == "random" else "centred 90x90 hole (49.4% unknown)",
           "parallelism": f"replicas x{args.gpus} (requests sharded, no data-path collective)",
           "l2": (f"inputs larger than L2, no flush: {touched:.0f} MB touched per sub-step launch vs 126 MB L2 (the "
                  "roofline probes additionally cycle 3 operand sets so every timed launch is L2-cold)")
                 if touched > 126 else f"working set {touched:.0f} MB fits L2; no flush"}
    if impl == "b200":
        cfg.update({"rng": args.rng, "jobs_per_step": args.jobs_per_step,
                    "api": "lanpaint_b200.comfy_nodes.LanPaint_KSampler.sample (ComfyUI replaced by minicomfy)"})
    return cfg


# ------------------------------------------------------------------------------------------
# node-API workloads
# ------------------------------------------------------------------------------------------
MASK_KIND = "random"


class Spec:
    """One benchmark configuration driven through LanPaint_KSampler.sample."""

    def __init__(self, name, batch, latent, n_inner=5, flow=False, shift=1.0, scheduler="karras", steps=N_OUTER,
                 cfg=5.0, note="", sampler="euler", network=None, model_type=None):
        self.name, self.batch, self.latent, self.n_inner, self.sampler = name, batch, tuple(latent), n_inner, sampler
        self.flow, self.shift, self.scheduler, self.steps, self.cfg, self.note = flow, shift, scheduler, steps, cfg, note
        self.network = network          # None: the pointwise synthetic network; else a torch module (minicomfy.networks)
        self.model_type = model_type    # None: FLOW / EPS from `flow`; "FLUX" sets cfg_BIG = 1 like the reference does

    @property
    def shape(self):
        return (self.batch,) + self.latent

    @property
    def n_el(self):
        n = self.batch
        for d in self.latent:
            n *= d
        return n


class NodeWorkload:
    def __init__(self, spec: Spec, dev, rng: str, seed: int = 0, extra_opts=None):
        import minicomfy
        minicomfy.install()
        from lanpaint_b200 import comfy_nodes as N
        from lanpaint_b200.runner import HostSchedule, SynthCondNet
        self.N, self.spec, self.dev, self.minicomfy = N, spec, dev, minicomfy
        g = torch.Generator().manual_seed(seed)
        shape = spec.shape
        y = torch.randn(shape, generator=g)
        mshape = (shape[0], 1) + tuple(shape[2:])
        if MASK_KIND == "blob" and len(shape) == 4:   # a real inpainting mask: one centred hole of ~half the area
            nm = torch.zeros(mshape)
            h, w = shape[2], shape[3]
            nm[:, :, int(0.15 * h):int(0.85 * h), int(0.15 * w):int(0.85 * w)] = 1.0
        else:                                           # SURVEY 8d: rand(B,1,*spatial) per site; 1 = regenerate
            nm = (torch.rand(mshape, generator=g) < 0.5).float()
        self.latent = {"samples": y.pin_memory(), "noise_mask": nm.pin_memory()}
        mtype = (getattr(minicomfy.ModelType, spec.model_type) if spec.model_type else
                 minicomfy.ModelType.FLOW if spec.flow else minicomfy.ModelType.EPS)
        self.net = spec.network if spec.network is not None else SynthCondNet()
        self.patcher = minicomfy.ModelPatcher(minicomfy.BaseModel(self.net, model_type=mtype, latent_channels=shape[1],
                                                                 shift=spec.shift), dev)
        opts = {"rng": rng, "timing": True}
        opts.update(extra_opts or {})
        self.patcher.model_options["lanpaint_b200"] = opts
        self.node = N.LanPaint_KSampler()
        sig = minicomfy.KSampler(self.patcher, spec.steps, dev, "euler", spec.scheduler).sigmas
        self.sched = HostSchedule([float(v) for v in sig], 1, spec.n_inner, spec.flow)
        self.substeps = self.sched.substeps
        self.guider_calls = self.sched.model_calls
        self.seed = 1000 * (seed + 1)
        self.h2d = (y.numel() * 2 + nm.numel()) * 4     # latent + ComfyUI's CPU noise image + the mask as it travels
        self.d2h = y.numel() * 4
        self.last_out = None

    def call(self):
        """One node call; returns (wall seconds, device ms of the sampler loop inside it)."""
        self.seed += 1
        t0 = time.perf_counter()
        (out,) = self.node.sample(self.patcher, self.seed, self.spec.steps, self.spec.cfg, self.spec.sampler,
                                  self.spec.scheduler, 0.3, -0.2, self.latent, 1.0, self.spec.n_inner, "Image First", "",
                                  self.N.IMAGE_MODE)
        wall = time.perf_counter() - t0            # the result is a host tensor: the call has synchronised
        e0, e1 = self.N.LAST_RUN["events"]
        if self.spec.sampler != "euler":           # other samplers evaluate the wrapper at sigmas of their own
            eng = self.N.LAST_ENGINE["engine"]
            self.substeps, self.guider_calls = eng.substeps_done, eng.model_calls
        self.last_out = out                        # the LATENT dict the caller receives
        return wall, e0.elapsed_time(e1)

    def warm(self, n=8):
        """eager -> capture (per-step graphs) -> replay -> [short job: capture the whole-job graph] -> replay;
        stops once two consecutive calls were pure replays of the same kind."""
        modes = []
        for _ in range(n):
            job = self.N.LAST_RUN.get("job")
            before = job.captures if job is not None else -1
            self.call()
            job = self.N.LAST_RUN.get("job")
            modes.append((self.N.LAST_RUN["mode"], job is not None and job.captures == before))
            if len(modes) >= 2 and modes[-1] == modes[-2] and modes[-1][1] and modes[-1][0] not in ("eager", None):
                break
        return self.N.LAST_RUN["mode"]

    def prepare_noise_ms(self, reps=3):
        """-> (ms of the noise image as THIS call draws it, ms of ComfyUI's own CPU prepare_noise, where it is drawn)."""
        best_cpu = float("inf")
        for k in range(reps):
            t0 = time.perf_counter()
            self.minicomfy.prepare_noise(self.latent["samples"], 7 + k)
            best_cpu = min(best_cpu, time.perf_counter() - t0)
        dev = self.N._noise_device(self.patcher)
        if dev is None:
            return 1e3 * best_cpu, 1e3 * best_cpu, "cpu (ComfyUI's prepare_noise)"
        from lanpaint_b200 import hostnoise
        best = float("inf")
        for k in range(reps + 1):
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            hostnoise.torch_cpu_randn(self.latent["samples"].size(), 7 + k, dev)
            torch.cuda.synchronize(dev)
            best = min(best, time.perf_counter() - t0)
        return 1e3 * best, 1e3 * best_cpu, "device (hostnoise.torch_cpu_randn: the bits of ComfyUI's CPU draw)"

    def stats(self):
        eng = self.N.LAST_ENGINE["engine"]
        job = self.N.LAST_RUN["job"]
        return {"mode": self.N.LAST_RUN["mode"], "fused_sampler": self.N.LAST_RUN["fused"],
                "graph_nodes_per_job": (eng.launches + 2 * eng.model_calls) if eng is not None else None,
                "graphs": job.captures if job is not None else None}


class OutputDump:
    """--dump-outputs: what the timed path handed back in its last step, so that two builds run with the same arguments
    can be compared output for output.  Every array of each call's LATENT dict is stacked over the step's calls and
    written as DIR/<key>.npy (float32).  When the whole step exceeds `budget` bytes, each call contributes the same fixed
    sample of flat element indices: the first n of torch.randperm(numel) under a generator seeded with 0, sorted."""

    def __init__(self, calls: int, budget: int = 60 * 10 ** 6):     # under 64 MB with the .npy headers
        self.calls, self.budget, self.rows, self.index = calls, budget, {}, {}

    def add(self, latent):
        arrays = {k: v for k, v in latent.items() if isinstance(v, torch.Tensor)}
        total = 4 * self.calls * sum(v.numel() for v in arrays.values())
        for key, v in arrays.items():
            v = v.detach().float().cpu()
            if total > self.budget:
                if key not in self.index:
                    n = v.numel() * self.budget // total
                    self.index[key] = torch.randperm(v.numel(), generator=torch.Generator().manual_seed(0))[:n].sort().values
                v = v.reshape(-1)[self.index[key]]
            self.rows.setdefault(key, []).append(v.clone())

    def write(self, out_dir: str):
        import numpy as np
        os.makedirs(out_dir, exist_ok=True)
        for key, rows in self.rows.items():
            np.save(os.path.join(out_dir, key + ".npy"), torch.stack(rows).numpy())


class DirectGuider:
    """The object the engine sees from ComfyUI's patched CFGGuider, without ComfyUI: cond / uncond evaluations of
    the same synthetic network, handed over as a CfgPair (both CFG combines happen in the update kernel)."""

    def __init__(self, net, sampling, cfg, cfg_big):
        self.inner_model, self.model_sampling, self.net, self.cfg, self.cfg_big = self, sampling, net, cfg, cfg_big

    def __call__(self, x, t, model_options=None, seed=None):
        from lanpaint_b200.engine import CfgPair
        return CfgPair(self.net(x, t, 0.3), self.net(x, t, -0.2), self.cfg, self.cfg_big)


def run_b200(args):
    import minicomfy
    from lanpaint_b200 import _native
    from lanpaint_b200.engine import LanPaint, pack_mask
    from lanpaint_b200.replicas import ReplicaGroup
    from lanpaint_b200.runner import (GraphedJob, HostSchedule, SynthCondNet, SynthDenoiser, VESampling, karras_sigmas,
                                      time_steady_substep)

    rank, world, local = dist_env()
    assert torch.cuda.is_available(), "bench.py (impl b200) needs a CUDA device; there is no CPU fallback"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa_node(local)
    group = ReplicaGroup(backend="nccl" if world > 1 else None, device=dev)   # init + barrier + max-over-ranks
    clocks = ClockSampler(local).start()
    minicomfy.install()
    R, K, W, J = args.requests, args.steps, max(3, args.warmup), args.jobs_per_step

    # replicas: the only collective is the one-time broadcast of the network's weights (north_star)
    weights = torch.tensor(SynthCondNet().coef, device=dev)
    group.broadcast_weights([weights])

    spec_main = Spec("sdxl_batch", R, SHAPE)
    other_rng = "philox" if args.rng == "torch" else "torch"

    def measure(spec, rng, steps, warm_steps, jobs, seed=rank, tag=None, dump=None):
        """steps x jobs node calls: device time of the sampler loops (sum, max over ranks) and wall time.  `dump`: an
        OutputDump that receives what each call of the last step returned."""
        wl = NodeWorkload(spec, dev, rng, seed=seed)
        wl.net.coef = tuple(weights.tolist())
        wl.warm()
        for _ in range(warm_steps * jobs):
            wl.call()
        wl.seed = 1000 * (seed + 1) + 10 ** 6     # timed calls draw the same seeds however many calls warming took
        group.barrier()
        if tag == "main":
            clocks.mark("t0")
        span_ms, wall_s = 0.0, 0.0
        for i in range(steps * jobs):
            w_, s_ = wl.call()
            wall_s += w_
            span_ms += s_
            if dump is not None and i >= (steps - 1) * jobs:
                dump.add(wl.last_out)             # outside call(): neither clock sees it
        group.barrier()
        if tag == "main":
            clocks.mark("t1")
        span_ms, wall_s = group.max_over_ranks(span_ms), group.max_over_ranks(wall_s)
        units = world * spec.batch * wl.substeps * steps * jobs
        st = wl.stats()
        rec = {"value": units / (span_ms * 1e-3), "ms_per_job_device": span_ms / (steps * jobs),
               "e2e_value": units / wall_s, "ms_per_job_wall": 1e3 * wall_s / (steps * jobs),
               "jobs": steps * jobs, "substeps_per_request": wl.substeps, "guider_calls_per_request": wl.guider_calls,
               "launch": st}
        return rec, wl

    # ---- main line: the node API at the shipped default -------------------------------------------------------
    dump = OutputDump(J) if args.dump_outputs and rank == 0 else None
    main, wl_main = measure(spec_main, args.rng, K, W, J, tag="main", dump=dump)
    if dump is not None:
        dump.write(args.dump_outputs)
    noise_ms, cpu_noise_ms, noise_where = wl_main.prepare_noise_ms()
    on_device = noise_where.startswith("device")
    wl_main.h2d = wl_main.h2d - (wl_main.latent["samples"].numel() * 4 if on_device else 0)   # no noise image to upload
    value, ms_per_step = main["value"], main["ms_per_job_device"] * J
    e2e = {"value": main["e2e_value"], "unit": "sub-steps/s", "h2d_bytes_per_step": wl_main.h2d * J,
           "d2h_bytes_per_step": wl_main.d2h * J, "steps": K, "jobs_per_step": J,
           "ms_per_job_wall": main["ms_per_job_wall"],
           "breakdown_ms_per_job": {"noise_image": noise_ms, "noise_image_drawn_on": noise_where,
                                    "comfyui_cpu_prepare_noise_it_replaces": cpu_noise_ms,
                                    "sampler_loop_on_device": main["ms_per_job_device"],
                                    "h2d_d2h_and_host_python": main["ms_per_job_wall"] - noise_ms - main["ms_per_job_device"]},
           "pcie_gbs": {"note": "latent + mask up (pageable CPU tensors as ComfyUI hands them over; the noise image too when "
                                "it is drawn on the CPU), result down through pinned memory",
                        "bytes_per_job": wl_main.h2d + wl_main.d2h},
           "numa_node": numa,
           "api": f"lanpaint_b200.comfy_nodes.LanPaint_KSampler.sample, rng={args.rng}, LATENT dict of host tensors in, LATENT "
                  "dict of host tensors out (every call: the noise image of comfy.sample.prepare_noise, H2D, sampler loop, D2H)"}
    # kernels of this repository launched inside the timed region: the job's graph nodes + the two noise-image kernels
    launches = ((wl_main.stats()["graph_nodes_per_job"] or 0) + (2 if on_device else 0)) * K * J * world

    # ---- secondary records: an exception in any of them is reported in the line, never in place of it ----------
    variants, serving, roofs, configs, other_sampler, real_network, frame_shard, cpu = {}, None, {}, None, None, None, None, None
    peak, peak_src = peaks()
    roof = {"bound": "hbm", "achieved": None, "peak": peak, "unit": "GB/s", "frac": None, "traffic": None,
            "peak_source": peak_src, "note": "kernel timer not run"}
    secondary_error = None
    try:
        # ---- rooflines: the steady fused sub-step of each stream (and with bf16 heads), live CUDA-event timing ------
        peak, peak_src = peaks()
        roofs = {}
        if args.kernel_timer:
            g = torch.Generator().manual_seed(90 + rank)
            y = torch.randn((R,) + SHAPE, generator=g).to(dev)
            known = (torch.rand((R, 1) + SHAPE[1:], generator=g) < 0.5).to(dev)
            pm = pack_mask(known, y)
            n_el = R * SHAPE[0] * SHAPE[1] * SHAPE[2]
            kernels = {"torch": ("lp::substep_torch_tma_kernel<float, first=0, next=1> (steady fused sub-step, torch.randn stream, "
                                 "producer warp + 4 plane slots of cp.async.bulk)", torch.float32),
                       "philox": ("lp::substep_tma_kernel<float, first=0, next=1, merge=1> (steady fused sub-step, philox stream, "
                                  "TMA-staged persistent)", torch.float32),
                       "torch_bf16_heads": ("lp::substep_torch_tma_kernel<bf16, first=0, next=1>", torch.bfloat16),
                       "philox_bf16_heads": ("lp::substep_tma_kernel<bf16, first=0, next=1, merge=1>", torch.bfloat16)}
            for key, (kname, hdtype) in kernels.items():
                rng = key.split("_")[0]
                eng = LanPaint(SynthDenoiser(VESampling(), dtype=hdtype), NSteps=N_INNER, Friction=15.0, Lambda=5.0, Beta=1.0,
                               StepSize=0.2, MinStepFrac=1.0, rng=rng, batched_replace="per_sample")
                algo = algo_bytes_per_elem(SHAPE[0], 4 if hdtype == torch.float32 else 2) * n_el
                burst = sorted(time_steady_substep(eng, y, pm, sigma=2.0, launches=53, repeats=20, rotate=3))
                avg = sum(burst) / len(burst)
                rec = {"bound": "hbm", "achieved": algo / (avg * 1e-6) / 1e9, "peak": peak, "unit": "GB/s",
                       "frac": algo / (avg * 1e-6) / 1e9 / peak, "traffic": None, "kernel": kname, "peak_source": peak_src,
                       "algorithmic_bytes_per_launch": algo, "avg_us": avg, "median_us": burst[len(burst) // 2],
                       "min_us": burst[0], "launches_timed": 53 * len(burst)}
                if key in ("torch", "philox"):
                    warm = sorted(time_steady_substep(eng, y, pm, sigma=2.0, launches=53, repeats=10, rotate=1))
                    rec["same_buffers_us"] = sum(warm) / len(warm)   # one operand set re-used: the L2 keeps part of it
                tr = os.path.join(ROOT, "profiles", "traffic.json")
                if os.path.exists(tr):
                    rec["traffic"] = json.load(open(tr)).get(f"{key}_{R}", json.load(open(tr)).get(str(R)) if key == "philox" else None)
                roofs[key] = rec
            roofs[args.rng]["timing"] = ("53 back-to-back launches of the steady fused sub-step between two CUDA events on the "
                                         "launching stream, x20, cycling 3 independent job-shaped operand sets so every launch's "
                                         "operands were evicted from L2 by the two launches before it (true HBM streaming)")
            roofs[args.rng]["substep_share_of_step"] = 53 * roofs[args.rng]["avg_us"] * 1e-3 / main["ms_per_job_device"]
            if rank == 0:
                # context for the fractions: the same copy probe MEASURED_PEAKS.json was produced with, on THIS box
                try:
                    a_ = torch.empty(1 << 30, dtype=torch.bfloat16, device=dev)
                    b_ = torch.empty_like(a_)
                    best = float("inf")
                    for _ in range(10):
                        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        c0.record()
                        b_.copy_(a_)
                        c1.record()
                        c1.synchronize()
                        best = min(best, c0.elapsed_time(c1))
                    roofs[args.rng]["copy_gbs_this_box"] = 2 * a_.numel() * 2 / (best * 1e-3) / 1e9
                    del a_, b_
                except Exception:
                    pass
            torch.cuda.empty_cache()
        roof = roofs.get(args.rng) or {"bound": "hbm", "achieved": None, "peak": peak, "unit": "GB/s", "frac": None,
                                       "traffic": None, "peak_source": peak_src}

        # ---- the other randn stream, same measurement (fewer steps) ------------------------------------------------
        variants = {}
        if not args.quick:
            v, _ = measure(spec_main, other_rng, max(2, K // 4), 1, J)
            variants[other_rng] = {"value": v["value"], "ms_per_job_device": v["ms_per_job_device"],
                                   "e2e": {"value": v["e2e_value"], "unit": "sub-steps/s", "ms_per_job_wall": v["ms_per_job_wall"],
                                           "api": f"lanpaint_b200.comfy_nodes.LanPaint_KSampler.sample, rng={other_rng}"},
                                   "jobs": v["jobs"], "launch": v["launch"]}

        # ---- serving path: runner.GraphedJob (host-owned sampler loop, whole job = one graph), same guider ---------
        serving = None
        if not args.quick:
            serving = {}
            sched = HostSchedule(karras_sigmas(N_OUTER), R, N_INNER)
            g = torch.Generator().manual_seed(50 + rank)
            y = torch.randn((R,) + SHAPE, generator=g).to(dev)
            noise = torch.randn((R,) + SHAPE, generator=g).to(dev)
            known = (torch.rand((R, 1) + SHAPE[1:], generator=g) < 0.5).to(dev)
            pm = pack_mask(known, y)
            for rng in (args.rng, other_rng):
                net = SynthCondNet(tuple(weights.tolist()))
                eng = LanPaint(DirectGuider(net, VESampling(), 5.0, 5.0), NSteps=N_INNER, Friction=15.0, Lambda=5.0, Beta=1.0,
                               StepSize=0.2, MinStepFrac=1.0, rng=rng, batched_replace="per_sample")
                job = GraphedJob(eng, sched, (R,) + SHAPE, dev)
                for _ in range(3):
                    job.run(y, noise, pm)
                group.barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                n_jobs = max(20, K)
                e0.record()
                for _ in range(n_jobs):
                    job.run(y, noise, pm)
                e1.record()
                group.barrier()
                ms = group.max_over_ranks(e0.elapsed_time(e1))
                serving[rng] = {"value": world * R * sched.substeps * n_jobs / (ms * 1e-3), "ms_per_job": ms / n_jobs,
                                "graph_nodes_per_job": job.launches + 2 * job.model_calls,
                                "api": "lanpaint_b200.runner.GraphedJob.run, device-resident inputs, one CUDA graph per job"}
                del job, eng
            # round 1's headline configuration for continuity: two-head synthetic network (ONE kernel per guider evaluation
            # instead of a cond and an uncond one), philox stream, whole-job graph
            eng = LanPaint(SynthDenoiser(VESampling()), NSteps=N_INNER, Friction=15.0, Lambda=5.0, Beta=1.0, StepSize=0.2,
                           MinStepFrac=1.0, rng="philox", batched_replace="per_sample")
            job = GraphedJob(eng, sched, (R,) + SHAPE, dev)
            for _ in range(3):
                job.run(y, noise, pm)
            group.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n_jobs):
                job.run(y, noise, pm)
            e1.record()
            group.barrier()
            ms = group.max_over_ranks(e0.elapsed_time(e1))
            serving["round1_headline_config"] = {"value": world * R * sched.substeps * n_jobs / (ms * 1e-3), "ms_per_job": ms / n_jobs,
                                                 "graph_nodes_per_job": job.launches + job.model_calls,
                                                 "what": "two-head synthetic network (73 network kernels per request instead of "
                                                         "146), rng=philox, runner.GraphedJob: the configuration of BENCH_r01.value"}
            del job, eng
            if world == 1:   # batch-size sweep of that configuration (R = 256: every byte from HBM; small R: launch-bound)
                sweep = []
                for r in (1, 8, 32, 64, 256):
                    s_r = HostSchedule(karras_sigmas(N_OUTER), r, N_INNER)
                    g_r = torch.Generator().manual_seed(5)
                    y_r = torch.randn((r,) + SHAPE, generator=g_r).to(dev)
                    n_r = torch.randn((r,) + SHAPE, generator=g_r).to(dev)
                    p_r = pack_mask((torch.rand((r, 1) + SHAPE[1:], generator=g_r) < 0.5).to(dev), y_r)
                    e_r = LanPaint(SynthDenoiser(VESampling()), NSteps=N_INNER, Friction=15.0, Lambda=5.0, Beta=1.0, StepSize=0.2,
                                   MinStepFrac=1.0, rng="philox", batched_replace="per_sample")
                    j_r = GraphedJob(e_r, s_r, (r,) + SHAPE, dev)
                    for _ in range(3):
                        j_r.run(y_r, n_r, p_r)
                    torch.cuda.synchronize()
                    reps = 40 if r <= 64 else 12
                    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a0.record()
                    for _ in range(reps):
                        j_r.run(y_r, n_r, p_r)
                    a1.record()
                    torch.cuda.synchronize()
                    t_r = a0.elapsed_time(a1) / reps
                    sweep.append({"requests_per_gpu": r, "ms_per_job": t_r, "value": r * s_r.substeps / (t_r * 1e-3),
                                  "us_per_graph_node": 1e3 * t_r / (j_r.launches + j_r.model_calls)})
                    del j_r, e_r, y_r, n_r, p_r
                    torch.cuda.empty_cache()
                serving["round1_headline_config"]["sweep"] = sweep
            ref_ms = serving[args.rng]["ms_per_job"]
            serving["node_api_over_graphed_job"] = main["ms_per_job_device"] / ref_ms
            # host tensors in, host result out through the same object, two batches in flight, uint8 mask, noise drawn on
            # the device (serving hosts do not need ComfyUI's CPU noise image): round 1's e2e, with less PCIe traffic
            lanes = []
            for lane in range(2):
                gl = torch.Generator().manual_seed(70 + rank + 17 * lane)
                hy = torch.randn((R,) + SHAPE, generator=gl).pin_memory()
                hm = (torch.rand((R, 1) + SHAPE[1:], generator=gl) < 0.5).to(torch.uint8).pin_memory()
                net = SynthCondNet(tuple(weights.tolist()))
                eng = LanPaint(DirectGuider(net, VESampling(), 5.0, 5.0), NSteps=N_INNER, Friction=15.0, Lambda=5.0, Beta=1.0,
                               StepSize=0.2, MinStepFrac=1.0, rng=args.rng, batched_replace="per_sample")
                lanes.append({"y": hy, "m": hm, "out": torch.empty((R,) + SHAPE).pin_memory(),
                              "stream": torch.cuda.Stream(device=dev), "job": GraphedJob(eng, sched, (R,) + SHAPE, dev)})

            def submit(ln):
                with torch.cuda.stream(ln["stream"]):
                    ln["job"].run(ln["y"], None, ln["m"].to(dev, non_blocking=True), x_out=ln["out"])

            def run_lanes(n):
                for i in range(n):
                    ln = lanes[i % 2]
                    ln["stream"].synchronize()      # the previous result of this lane is on the host: the user has it
                    submit(ln)
                for ln in lanes:
                    ln["stream"].synchronize()
            run_lanes(6)
            group.barrier()
            n_jobs = max(20, K)
            t0 = time.perf_counter()
            run_lanes(n_jobs)
            group.barrier()
            dt = group.max_over_ranks(time.perf_counter() - t0)
            bi = lanes[0]["y"].numel() * 4 + lanes[0]["m"].numel()
            bo = lanes[0]["out"].numel() * 4
            serving["e2e"] = {"value": world * R * sched.substeps * n_jobs / dt, "unit": "sub-steps/s",
                              "h2d_bytes_per_job": bi, "d2h_bytes_per_job": bo, "jobs": n_jobs, "in_flight": 2,
                              "pcie_gbs": {"h2d": bi * n_jobs / dt / 1e9, "d2h": bo * n_jobs / dt / 1e9},
                              "api": f"lanpaint_b200.runner.GraphedJob.run(latent pinned host, noise=None (drawn on the device), "
                                     f"uint8 mask pinned host) -> pinned host result, rng={args.rng}"}
            del lanes

        # ---- the literal BASELINE configurations, each through the node API ------------------------------------------
        configs = None
        specs = [Spec("cfg2_sdxl_batch1_N5", 1, SHAPE, note="BASELINE configs[1]"),
                 Spec("sdxl_batch8_N5", 8, SHAPE, note="north_star target shape"),
                 Spec("cfg3_sdxl_4_per_gpu_N10", 4, SHAPE, n_inner=10, note="BASELINE configs[2]: batch 32 = 4 per GPU x 8"),
                 Spec("cfg4_flux_16x128x128_flow_simple20", 1, (16, 128, 128), flow=True, shift=1.0, scheduler="simple",
                      cfg=1.0 + 2.5, note="BASELINE configs[3] at the ComfyUI boundary (patchify is inside the DiT)"),
                 Spec("cfg5_wan_16x21x80x45_flow_simple20_shift3", 1, (16, 21, 80, 45), flow=True, shift=3.0, scheduler="simple",
                      note="BASELINE configs[4], 81 frames -> 21 latent frames, one GPU holds the sample (see --frame-shard)")]
        if args.configs and not args.quick:
            configs = []
            for sp in specs:
                if world > 1 and not sp.name.startswith("cfg3"):
                    continue           # SCALE carries cfg3 (32 requests over 8 GPUs); the rest are single-GPU records
                recs = {}
                for rng in (args.rng, other_rng):
                    r_, wl = measure(sp, rng, 1, 0, 12 if sp.batch <= 8 else 6, seed=rank + 3)
                    recs[rng] = r_
                r0 = recs[args.rng]
                c = {"name": sp.name, "note": sp.note, "latent_shape": list(sp.shape), "think_steps": sp.n_inner,
                     "schedule": f"{sp.scheduler}-{sp.steps}" + (f" shift {sp.shift}" if sp.flow else ""),
                     "substeps": r0["substeps_per_request"], "guider_calls": r0["guider_calls_per_request"],
                     "n_gpus": world, "api": "comfy_nodes.LanPaint_KSampler.sample"}
                for rng, r_ in recs.items():
                    nodes = r_["launch"]["graph_nodes_per_job"]
                    algo = algo_bytes_per_elem(sp.latent[0]) * sp.n_el * r_["substeps_per_request"]
                    c[rng] = {"value": r_["value"], "ms_per_job_device": r_["ms_per_job_device"], "e2e_value": r_["e2e_value"],
                              "ms_per_job_wall": r_["ms_per_job_wall"], "launch_mode": r_["launch"]["mode"],
                              "graph_nodes_per_job": nodes,
                              "us_per_graph_node": 1e3 * r_["ms_per_job_device"] / nodes if nodes else None,
                              "substep_algorithmic_gbs": algo / (r_["ms_per_job_device"] * 1e-3) / 1e9,
                              "regime": "latency / L2 (working set %.1f MB per launch)" % (5.25 * 4 * sp.n_el / 1e6)}
                if rank == 0 and world == 1:
                    c["reference_eager_on_this_gpu"] = eager_reference_on_gpu(sp, dev)
                    if c["reference_eager_on_this_gpu"].get("ms_per_job"):
                        c["speedup_vs_reference_on_this_gpu"] = (c["reference_eager_on_this_gpu"]["ms_per_job"] /
                                                                c[args.rng]["ms_per_job_device"])
                configs.append(c)
                torch.cuda.empty_cache()

        # ---- another sampler through the same node: k-diffusion's own loop captured as one graph ---------------------
        other_sampler = None
        if args.configs and not args.quick and world == 1:
            rec, wl = measure(Spec("sdxl_batch_heun", R, SHAPE, sampler="heun"), args.rng, 1, 0, 8, seed=rank + 7)
            other_sampler = {"sampler": "heun", "requests_per_gpu": R, "value": rec["value"],
                             "ms_per_job_device": rec["ms_per_job_device"], "e2e_value": rec["e2e_value"],
                             "substeps_per_request": rec["substeps_per_request"],
                             "guider_calls_per_request": rec["guider_calls_per_request"], "launch": rec["launch"],
                             "note": "heun evaluates the wrapper twice per step; its whole loop (k-diffusion's Python) is captured "
                                     "into one CUDA graph after an eager first job recorded the sigma sequence"}
            del wl
            torch.cuda.empty_cache()

        # ---- cfg4 with a real PyTorch network captured in the graphs -------------------------------------------------
        real_network = None
        if args.real_network and not args.quick and world == 1:
            try:
                real_network = run_real_network(dev, args)
            except Exception as e:   # an informational record never breaks the bench line
                real_network = {"error": f"{type(e).__name__}: {e}"}

        # ---- cfg5 frame-sharded synthetic run: one sample's frames split over the ranks ------------------------------
        frame_shard = None
        if args.frame_shard and not args.quick:
            frame_shard = run_frame_shard(group, dev, args)

        # ---- CPU baseline: the reference on the host cores, bounded sample (rank 0, N=1 only) ----
        cpu = None
        if rank == 0 and world == 1 and not args.no_cpu:
            import warnings
            warnings.filterwarnings("ignore")
            host_cores = os.cpu_count() or 1
            kind = reference_engine_kind()
            ref_nodes = reference_nodes() if kind == "reference" else None
            cores = calibrate_threads(args.ref_requests)
            cpu_job(2, 2, cores)  # warm
            if ref_nodes is not None:
                dt, u = cpu_node_job(ref_nodes, args.ref_requests, cores)
            else:
                dt, u = cpu_job(args.ref_requests, N_OUTER, cores)
            cpu = {"value": u / dt, "unit": "sub-steps/s", "cores": cores, "kind": kind,
                   "same_reference_math_on_this_gpu": eager_reference_on_gpu(Spec("sdxl_batch8", args.ref_requests, SHAPE), dev),
                   "sample": f"{args.ref_requests} of {R} requests, full karras-20 x N=5 schedule, {dt:.1f} s of CPU work; "
                             f"{cores} torch threads (fastest of a probe over 1..{host_cores} host cores); "
                             + (REFERENCE_API if ref_nodes is not None else
                                "engine = the reference's own LanPaint.__call__ (oracle/_ref bytecode)" if kind == "reference"
                                else "oracle port")}

    except Exception as e:
        if world > 1:      # the other ranks are inside collectives of the same section: fail fast instead of hanging them
            raise
        import traceback
        secondary_error = f"{type(e).__name__}: {e} @ " + traceback.format_exc().strip().splitlines()[-3].strip()

    clocks.stop()
    if rank == 0:
        cfg = workload_config(args)
        cfg["timing"] = ("value: sum over the timed calls of the device time between two CUDA events the node layer records "
                         "inside KSAMPLER.sample (inputs on the device -> last kernel of the sampler loop), barrier + "
                         "synchronize on both sides of the timed region, max over ranks; e2e: wall clock of the same calls")
        cfg["launch"] = main["launch"]
        if configs is not None:
            cfg["configs"] = configs
        line = {
            "metric": METRIC, "value": value, "unit": "sub-steps/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg, "roofline": roof, "rooflines": roofs, "cpu_baseline": cpu, "e2e": e2e,
            "variants": variants, "serving": serving, "frame_shard": frame_shard, "other_sampler": other_sampler,
            "real_network": real_network, "secondary_error": secondary_error,
            "gpu_launches": launches, "clocks": clocks.summary(),
        }
        print(json.dumps(line), flush=True)
    group.close()


def eager_reference_on_gpu(spec: Spec, dev, model=None):
    """The reference's math (oracle port, op for op) with device="cuda": what a user of the reference runs today on
    this very GPU (eager PyTorch, ~89 element-wise launches per sub-step).  Informational, not the reference arm.
    `model`: a guider double around a real network (default: the oracle's pointwise two-head network)."""
    try:
        from oracle import langevin_oracle as O
        import minicomfy
        g = torch.Generator().manual_seed(3)
        shape = spec.shape
        y = torch.randn(shape, generator=g).to(dev)
        noise = torch.randn(shape, generator=g).to(dev)
        dm = (torch.rand((shape[0], 1) + tuple(shape[2:]), generator=g) < 0.5).float().to(dev).expand(shape).contiguous()
        if spec.flow:
            sig = minicomfy.simple_scheduler(minicomfy.ModelSamplingCONST(spec.shift), spec.steps).to(dev)
            sampling = O.FlowSampling()
        else:
            sig = O.karras_sigmas(spec.steps).to(dev)
            sampling = O.VESampling()
        hp = O.Hyper(n_steps=spec.n_inner, min_step_frac=1.0, flow=spec.flow)
        cnt = {}
        if model is None:
            model = O.PointwiseDenoiser(sampling)
        else:
            model.model_sampling = sampling
        with torch.no_grad():
            O.euler_inpaint(model, y, noise, dm, sig, hp, counters=cnt)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            O.euler_inpaint(model, y, noise, dm, sig, hp, counters=cnt)
            torch.cuda.synchronize()
        tq = time.perf_counter() - t0
        return {"value": shape[0] * cnt["substeps"] / tq, "unit": "sub-steps/s", "requests": shape[0],
                "ms_per_job": 1e3 * tq, "what": "oracle port, device=cuda, eager launches, same schedule"}
    except Exception as e:  # never let the informational leg break the bench line
        return {"error": f"{type(e).__name__}: {e}"}


class NetworkGuider:
    """What the reference's patched CFGGuider hands its engine when cfg == 1 (Flux: uncond skipped, cfg_BIG = 1):
    both heads are the one conditional evaluation of the network (nodes.py:161-175, 331-334)."""

    def __init__(self, net, cond):
        self.inner_model, self.model_sampling, self.net, self.cond = self, None, net, cond

    def __call__(self, x, t, model_options=None, seed=None):
        out = self.net(x, t, self.cond)
        return out, out


def run_real_network(dev, args):
    """BASELINE configs[3] with a real PyTorch network in the loop: a Flux-shaped bf16 DiT stand-in (random weights;
    minicomfy.networks.DiTStandIn) behind `LanPaint_KSampler.sample`, [1,16,128,128] latent, flow simple-20 x N=5,
    cfg 1 (52 sub-steps, 72 forwards per job).  The node path captures the network together with the update kernels
    (north_star: "CUDA-graph-captured once per (shape, sigma) and replayed inside the inner loop"); reported next to
    plain launches of the same path and to the reference's math run eagerly around the same network on this GPU."""
    from minicomfy.networks import DiTStandIn
    torch.manual_seed(1234)
    net = DiTStandIn().to(dev).eval()
    spec = Spec("cfg4_flux_dit", 1, (16, 128, 128), flow=True, shift=1.15, scheduler="simple", cfg=1.0,
                network=net, model_type="FLUX")
    out = {"network": f"minicomfy.networks.DiTStandIn: 2x2 patchify -> 4096 tokens, hidden {net.hidden}, "
                      f"{len(net.blocks)} adaLN blocks, bf16 SDPA attention, {net.n_params() / 1e6:.0f} M random-init parameters, "
                      "x0 = x - sigma * v in fp32 (ComfyUI's calculate_denoised)",
           "latent": [1, 16, 128, 128], "schedule": "flow simple-20 shift 1.15, N=5, cfg 1.0 (uncond skipped, cfg_BIG = 1)"}
    with torch.no_grad():
        x = torch.randn(1, 16, 128, 128, device=dev)
        t = torch.full((1,), 0.5, device=dev)
        for _ in range(3):
            net(x, t, 0.3)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            net(x, t, 0.3)
        e1.record()
        e1.synchronize()
        out["network_forward_ms_eager"] = e0.elapsed_time(e1) / 10
        # the same ten forwards as one CUDA graph: what a forward costs inside the captured job
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.stream(side):
            with torch.cuda.graph(graph, stream=side):
                for _ in range(10):
                    net(x, t, 0.3)
        torch.cuda.current_stream(dev).wait_stream(side)
        graph.replay()
        e0.record()
        graph.replay()
        e1.record()
        e1.synchronize()
        fwd_ms = e0.elapsed_time(e1) / 10
        out["network_forward_ms_graph_replay"] = fwd_ms
        del graph
        for key, opts in (("graph_replay", {}), ("plain_launches", {"cuda_graph": False})):
            wl = NodeWorkload(spec, dev, args.rng, seed=5, extra_opts=opts)
            for _ in range(3):          # eager -> capture -> replay
                wl.call()
            n, wall, span = 3, 0.0, 0.0
            for _ in range(n):
                w_, s_ = wl.call()
                wall += w_
                span += s_
            st = wl.stats()
            st.pop("graph_nodes_per_job", None)      # that count assumes the one-kernel synthetic network
            out[key] = {"ms_per_job_device": span / n, "ms_per_job_wall": 1e3 * wall / n, "launch": st,
                        "substeps": wl.substeps, "network_forwards": wl.guider_calls,
                        "substeps_per_s": wl.substeps / (span / n * 1e-3)}
            del wl
        calls0 = net.calls
        out["reference_math_eager_on_this_gpu"] = eager_reference_on_gpu(spec, dev, NetworkGuider(net, 0.3))
        out["reference_math_eager_on_this_gpu"]["network_forwards_per_job"] = (net.calls - calls0) // 2
    g = out["graph_replay"]
    out["update_path_share_of_job"] = max(0.0, 1.0 - g["network_forwards"] * fwd_ms / g["ms_per_job_device"])
    ref = out["reference_math_eager_on_this_gpu"]
    if "ms_per_job" in ref:
        out["speedup_vs_reference_math_eager"] = ref["ms_per_job"] / g["ms_per_job_wall"]
        out["note"] = ("with a real network the job is the network: the update path's share is what is left after "
                       "network_forwards x network_forward_ms_graph_replay; the reference spends its extra time on ~89 eager launches "
                       "per sub-step and 2 + N + 1 host read-backs per outer step")
    del net
    torch.cuda.empty_cache()
    return out


def run_frame_shard(group, dev, args):
    """BASELINE configs[4] in its synthetic form (SURVEY 8e row 2): ONE Wan sample [1,16,21,80,45], its 21 latent
    frames split over the ranks; the update kernels need no exchange, the early stopper's two masked sums are the
    only cross-shard quantity (one all_reduce of 2 doubles per check)."""
    from lanpaint_b200.frame_shard import FrameShardedRun
    out = {}
    for key, thr in (("stopper_off", 0.0), ("stopper_on", args.frame_shard_threshold)):
        try:
            run = FrameShardedRun(group, dev, latent=(16, 21, 80, 45), n_inner=N_INNER, steps=N_OUTER, shift=3.0,
                                  early_stop_threshold=thr)
            out[key] = run.bench(jobs=10 if thr <= 0 else 3)
        except Exception as e:
            out[key] = {"error": f"{type(e).__name__}: {e}"}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--requests", type=int, default=128, help="independent SDXL requests batched per GPU")
    ap.add_argument("--jobs-per-step", type=int, default=16,
                    help="node calls per bench step (16 x ~3.5 ms of device time x 20 steps > 1 s timed)")
    ap.add_argument("--ref-requests", type=int, default=8, help="requests per step in the CPU arm's bounded sample")
    ap.add_argument("--rng", default="torch", choices=["philox", "torch"],
                    help="torch (default, what the nodes ship: the reference's own randn stream) | philox")
    ap.add_argument("--quick", action="store_true", help="main line + rooflines only")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-configs", dest="configs", action="store_false", help="skip the BASELINE configuration records")
    ap.add_argument("--no-kernel-timer", dest="kernel_timer", action="store_false")
    ap.add_argument("--no-frame-shard", dest="frame_shard", action="store_false")
    ap.add_argument("--no-real-network", dest="real_network", action="store_false",
                    help="skip the cfg4 record with the bf16 DiT stand-in in the loop")
    ap.add_argument("--frame-shard-threshold", type=float, default=0.05,
                    help="InnerThreshold of the frame-sharded record that runs with the early stopper on")
    ap.add_argument("--mask", default="random", choices=["random", "blob"],
                    help="random 50%% per site (SURVEY 8d, default) | one centred hole of about the same area")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the main line's last timed step returned as DIR/<key>.npy (float32, <= 64 MB in "
                         "all; a fixed seeded sample when larger); rank 0 only, b200 impl only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    global MASK_KIND
    MASK_KIND = args.mask
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
