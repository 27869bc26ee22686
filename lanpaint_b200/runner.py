"""Host-scheduled sampling runs over the engine (SURVEY 8f rank 3).

`HostSchedule` does on the host, once per run, what the reference's per-sigma
wrapper recomputes on the device every outer step with two syncs
(src/LanPaint/nodes.py:242-252,286-299): the (VE sigma, abt, flow t) triple and
the effective inner-step count for every sigma of the schedule.
`euler_inpaint` is then the reference's `LanPaint_KSampler` run with sampler
"euler" (nodes.py:338,376-378 around k-diffusion's sample_euler) expressed as a
sync-free launch sequence.

`SynthDenoiser` is the SURVEY 8d pointwise two-head stand-in for the UNet/DiT,
running as one CUDA kernel (lp_synth_denoiser_f32); bench.py and the tests use it.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import List, Optional, Sequence

import torch

from . import _native
from .schedule import effective_inner_steps, times_from_sigma


class VESampling:
    """EPS-type model_sampling: noise_scaling = y + sigma*noise (what nodes.py:338 relies on)."""

    def noise_scaling(self, sigma, noise, latent_image, max_denoise=False):
        if max_denoise:
            return noise * torch.sqrt(1.0 + sigma ** 2.0) + latent_image
        return latent_image + noise * sigma

    def inverse_noise_scaling(self, sigma, latent):
        return latent


class FlowSampling:
    """CONST-type (rectified flow) model_sampling."""

    noise_scale = 1.0

    def noise_scaling(self, sigma, noise, latent_image, max_denoise=False):
        return sigma * (self.noise_scale * noise) + (1.0 - sigma) * latent_image

    def inverse_noise_scaling(self, sigma, latent):
        return latent / (1.0 - sigma)


class SynthDenoiser:
    """x -> (a0 x + b0 tanh x + c0, a1 x + c1) as ONE kernel writing both heads.

    Follows the model protocol of the engine seam (`inner_model.model_sampling`,
    `__call__(x, t, model_options=, seed=)`).  Output buffers are reused, which is
    what a CUDA-graph-captured network does too."""

    def __init__(self, sampling=None, coef=(0.7, 0.1, 0.0, 0.6, -0.05), two_heads: bool = True,
                 dtype: torch.dtype = torch.float32):
        self.inner_model = self
        self.model_sampling = sampling or VESampling()
        self.coef = tuple(float(c) for c in coef)
        self._coef_c = (C.c_float * 5)(*self.coef)
        self.two_heads = two_heads
        self.dtype = dtype     # element type of the returned heads (a network computing in bf16 returns bf16)
        self._dtype_code = {torch.float32: _native.DTYPE_F32, torch.bfloat16: _native.DTYPE_BF16,
                            torch.float16: _native.DTYPE_F16}[dtype]
        self.calls = 0
        self._h0: Optional[torch.Tensor] = None
        self._h1: Optional[torch.Tensor] = None
        self._lib = _native.load()

    def set_coef(self, coef: Sequence[float]):
        self.coef = tuple(float(c) for c in coef)
        self._coef_c = (C.c_float * 5)(*self.coef)

    def __call__(self, x, t, model_options=None, seed=None):
        if self._h0 is None or self._h0.shape != x.shape or self._h0.device != x.device:
            self._h0 = torch.empty_like(x, dtype=self.dtype)
            self._h1 = torch.empty_like(x, dtype=self.dtype) if self.two_heads else None
        rc = self._lib.lp_synth_denoiser(C.c_void_p(x.data_ptr()), C.c_void_p(self._h0.data_ptr()),
                                         C.c_void_p(self._h1.data_ptr()) if self._h1 is not None else None,
                                         self._dtype_code, x.numel(), self._coef_c,
                                         C.c_void_p(torch.cuda.current_stream(x.device).cuda_stream))
        _native.check(rc, "lp_synth_denoiser")
        self.calls += 1
        return (self._h0, self._h1) if self.two_heads else self._h0


class SynthCondNet:
    """`denoiser(x, sigma, cond) -> x0` for a ComfyUI-style BaseModel (bench / tests): the same pointwise
    kernel as SynthDenoiser, one head per call, `cond` (a float standing in for CONDITIONING) shifts the
    output.  One output buffer per distinct cond, reused across calls like a captured network's."""

    def __init__(self, coef=(0.7, 0.1, 0.0)):
        self.coef = tuple(float(c) for c in coef)
        self._out = {}
        self._lib = _native.load()
        self.calls = 0

    def __call__(self, x, sigma, cond):
        c = float(cond)
        key = (c, tuple(x.shape), x.device)
        out = self._out.get(key)
        if out is None:
            out = self._out[key] = (torch.empty_like(x), (C.c_float * 5)(self.coef[0], self.coef[1], self.coef[2] + c, 0.0, 0.0))
        rc = self._lib.lp_synth_denoiser_f32(C.c_void_p(x.data_ptr()), C.c_void_p(out[0].data_ptr()), None, x.numel(),
                                             out[1], C.c_void_p(torch.cuda.current_stream(x.device).cuda_stream))
        _native.check(rc, "lp_synth_denoiser_f32")
        self.calls += 1
        return out[0]


@dataclass
class OuterStep:
    sigma: float
    sigma_next: float
    n_inner: int
    sigma_t: torch.Tensor    # CPU [B] fp32, what the sampler would pass as `sigma`
    times: tuple             # CPU (VE_Sigma, abt, Flow_t), reference op order (nodes.py:242-252)


class HostSchedule:
    """All per-sigma scalars of a run, computed once on the host."""

    def __init__(self, sigmas: Sequence[float], batch: int, n_inner: int, flow: bool = False,
                 early_stop: int = 1, min_step_frac: float = 1.0):
        sig = torch.as_tensor(list(sigmas), dtype=torch.float32)
        self.sigmas = sig
        host = [float(v) for v in sig]
        self.steps: List[OuterStep] = []
        ones = torch.ones(batch, dtype=torch.float32)
        for i in range(len(host) - 1):
            s = sig[i] * ones
            tm = times_from_sigma(s, flow)
            n_eff = effective_inner_steps(n_inner, host, float(torch.mean(s)), float((1.0 - tm[1]).mean()),
                                          early_stop, min_step_frac)
            self.steps.append(OuterStep(host[i], host[i + 1], n_eff, s, tm))
        self.substeps = sum(st.n_inner for st in self.steps)
        self.model_calls = self.substeps + len(self.steps)


def karras_sigmas(n: int, sigma_min: float = 0.0292, sigma_max: float = 14.6146, rho: float = 7.0) -> List[float]:
    """SDXL's karras schedule (SURVEY 8d), trailing 0 included."""
    ramp = torch.linspace(0, 1, n, dtype=torch.float32)
    lo, hi = sigma_min ** (1 / rho), sigma_max ** (1 / rho)
    s = (hi + ramp * (lo - hi)) ** rho
    return [float(v) for v in s] + [0.0]


def euler_inpaint(engine, latent_image: torch.Tensor, noise: torch.Tensor, mask, sched: HostSchedule,
                  x_out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """One full inpaint job on device-resident inputs; returns the final latent.

    mask: latent_mask (1 = known) tensor or an engine PackedMask."""
    sampling = engine.inner_model.inner_model.model_sampling
    x = sampling.noise_scaling(sched.sigmas[0].to(latent_image.device), noise, latent_image)
    for st in sched.steps:
        denoised = engine(x, latent_image, noise, st.sigma_t, mask, st.times, None, 0, n_steps=st.n_inner)
        # k-diffusion sample_euler: d = (x - denoised)/sigma ; x = x + d*(sigma_next - sigma)
        x = torch.add(x, x - denoised, alpha=(st.sigma_next - st.sigma) / st.sigma)
    if x_out is not None:
        x_out.copy_(x, non_blocking=True)
        return x_out
    return x


def time_steady_substep(engine, latent_image: torch.Tensor, mask, sigma: float, launches: int = 53,
                        repeats: int = 20, flow: bool = False, rotate: int = 3):
    """Roofline probe: `launches` steady fused sub-step launches (flags = FUSE_NEXT, the kernel that
    dominates a job) back to back on job-shaped operands, between two CUDA events on the launching
    stream, `repeats` times.  Returns the list of per-launch durations in microseconds (one per repeat).

    `rotate` independent operand sets (x, x0, x0_BIG, y, C, mask) are cycled, so a launch's operands were
    last touched `rotate - 1` launches ago: with 176 MB per set at the bench's default size that is far more
    than the 126 MB L2 can hold, i.e. every launch really streams from HBM (rotate=1 re-uses one set and lets
    the L2 keep part of it -- reported separately as the L2-assisted figure).  The launches are identical to
    those `LanPaint._launch_sequence` issues, minus the model call between them."""
    import numpy as np
    from .engine import PackedMask, _DrawPlan, pack_mask
    from .schedule import Hyper, build_table
    lib = _native.load()
    dev = latent_image.device
    B = latent_image.shape[0]
    pm0 = mask if isinstance(mask, PackedMask) else pack_mask(mask, latent_image)
    sets = []
    for r in range(max(1, rotate)):
        x = torch.randn_like(latent_image)
        heads = engine.inner_model(x, torch.full((B,), sigma, device=dev))
        x0, x0b = engine.unpack_model_output(heads)
        sets.append(dict(x=x, x0=x0.clone(), x0b=x0b.clone(), y=latent_image if r == 0 else latent_image.clone(),
                         c=torch.randn_like(x), m=pm0.data if r == 0 else pm0.data.clone()))
    s = torch.full((B,), sigma, dtype=torch.float32)
    ve, abt, _ = times_from_sigma(s, flow)
    hp = Hyper(engine.step_size, engine.chara_lamb, engine.chara_beta, engine.min_step_frac, flow)
    tab = torch.from_numpy(build_table(abt.numpy(), ve.numpy(), hp)).to(dev)
    per_row = latent_image.numel() // B
    spatial = int(np.prod(latent_image.shape[2:]))
    dims = _native.Dims(B, per_row, spatial, pm0.row_stride, pm0.channel_stride)
    plan = _DrawPlan(engine.rng, latent_image, launches + 1)
    merge = plan.mode == _native.RNG_PHILOX and engine.merge_noise
    flags = _native.SUBSTEP_FUSE_NEXT | (_native.SUBSTEP_MERGE_NOISE if merge else 0)
    P = C.c_void_p
    stream = P(torch.cuda.current_stream(dev).cuda_stream)

    from .engine import _heads
    for o in sets:   # heads in whatever dtype the model returns (fp32 / bf16 / fp16)
        o["heads"], o["keep"] = _heads(o["x0"], o["x0b"], o["x"])

    def burst():
        for k in range(launches):
            o = sets[k % len(sets)]
            r = plan.rng_struct(1 if merge else 2)
            rc = lib.lp_substep(P(o["x"].data_ptr()), C.byref(o["heads"]), P(o["y"].data_ptr()), P(o["m"].data_ptr()),
                                P(o["c"].data_ptr()), None, None, P(tab.data_ptr()), C.byref(dims), C.byref(r), flags,
                                stream)
            _native.check(rc, "lp_substep")

    for _ in range(3):
        burst()
    torch.cuda.synchronize(dev)
    out = []
    for _ in range(repeats):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        burst()
        e1.record()
        e1.synchronize()
        out.append(1e3 * e0.elapsed_time(e1) / launches)
    return out


class GraphedJob:
    """A whole inpaint job -- initial noise_scaling, every outer step (prologue, model calls, fused
    sub-steps, epilogue) and the Euler updates between them -- on static buffers, launched in one of
    three ways that share ONE body (`_step`):

      mode "job"    the whole job is ONE CUDA graph (captured once, replayed per batch of requests); with a callback
                    every outer step writes its denoised latent to its own buffer and the callbacks run, in order,
                    after the replay (for jobs so short that nobody can watch a progress bar move);
      mode "steps"  one CUDA graph per outer step, replayed in order with a host callback between them
                    (ComfyUI's progress / preview callback wants the denoised latent of every step);
      mode "eager"  plain launches (the first job of a configuration: nothing is wasted on warm-up).

    Everything sigma-dependent is a device constant computed at construction (one coefficient table per
    outer step), so a replay costs one 16-byte H2D copy (the RNG position) plus the copies of the
    request's own inputs.  Used directly by hosts that own the sampler loop (serving: fixed schedule,
    fixed batch shape, a stream of request batches) and by the node path (`comfy_nodes.KSAMPLER.sample`)
    whenever the ComfyUI sampler is plain Euler, the configuration the reference recommends
    (src/LanPaint/nodes.py:459 "Recommended: euler").

    Semantics are exactly `euler_inpaint(engine, ...)`, i.e. k-diffusion's sample_euler around the
    per-sigma wrapper (asserted bit-for-bit by the tests)."""

    def __init__(self, engine, sched: HostSchedule, shape, device, flow: bool = False, fused_euler: bool = True,
                 model_options=None, seed=0, external_init: bool = False, first_replace_noop=None):
        import numpy as np
        from .engine import _DrawPlan
        self.fused_euler = fused_euler   # Euler update inside lp_epilogue_euler_f32 instead of two torch kernels
        from .schedule import Hyper, build_table, mean_half_dt
        if engine.rng not in ("philox", "torch"):
            raise ValueError("GraphedJob needs an in-kernel RNG mode ('philox' or 'torch')")
        self.engine, self.sched, self.flow = engine, sched, flow
        self.model_options, self.seed = model_options, seed
        self.external_init = external_init   # run(x_init=...) supplies the initial state (node path: max_denoise etc.)
        self.device = torch.device(device)
        self.shape = tuple(shape)
        B = self.shape[0]
        dev = self.device
        mk = lambda: torch.empty(self.shape, dtype=torch.float32, device=dev)
        self.x, self.y, self.noise, self.c, self.out = mk(), mk(), mk(), mk(), mk()
        self.mask = None
        hyper = Hyper(engine.step_size, engine.chara_lamb, engine.chara_beta, engine.min_step_frac, flow)
        tabs, tms, sgs, self.active = [], [], [], []
        for st in sched.steps:
            ve, abt, flow_t = (t.numpy() for t in st.times)
            sig = st.sigma_t.numpy()
            form = engine._replace_form(sig, st.sigma_t.numel() == 1, B, engine.replace_mode, engine.batched_replace)
            if form is None:
                raise ValueError("model_sampling.noise_scaling is not a linear form; GraphedJob cannot precompute it")
            tabs.append(build_table(abt, ve, hyper, form[0], form[1]))
            tms.append(flow_t if flow else ve)
            sgs.append(sig)
            self.active.append(st.n_inner if mean_half_dt(abt, hyper) > 0.0 else 0)
        # draws consumed before outer step i (1 for sub-step 0, 2 for each later one): lets every outer step be
        # captured on its own against ONE {seed, base} block that is refreshed once per job
        merged = engine.rng == "philox" and engine.merge_noise   # a fused launch then draws ONE normal, not two
        self.draws_before = [0]
        for n in self.active:
            self.draws_before.append(self.draws_before[-1] + (0 if n <= 0 else (n if merged else 2 * n - 1)))
        self.tables = torch.from_numpy(np.stack(tabs)).to(dev)
        self.t_model = torch.from_numpy(np.stack(tms).astype(np.float32)).to(dev)
        self.sigma = torch.from_numpy(np.stack(sgs).astype(np.float32)).to(dev)
        self.sigma0 = torch.tensor(float(sched.sigmas[0]), device=dev)
        self.rng_state = torch.zeros(2, dtype=torch.int64, device=dev)
        if first_replace_noop is None:
            # the first replace step is a no-op when the replace form is noise_scaling's own form at sigmas[0]
            # (every known position of x already holds it); the reference's batched flow-form quirk differs
            first_replace_noop = (not external_init) and (B == 1 or engine.batched_replace == "per_sample")
        self.first_replace_noop = bool(first_replace_noop) and fused_euler
        self._graphs = {}
        self._dims = None
        self.timing, self.last_events = False, None
        self.outs = None     # per-outer-step denoised latents (mode "job" with a callback: callbacks run after the replay)
        self.launches = 0
        self.model_calls = 0
        self.captures = 0
        self._plan_cls = _DrawPlan

    @property
    def draws(self) -> int:
        return self.draws_before[-1]

    @property
    def graph(self):
        """The whole-job graph (None until the first mode="job" run)."""
        return self._graphs.get(("job", False))

    def per_step_bytes(self) -> int:
        return len(self.sched.steps) * self.x.numel() * 4

    # ---- the body ------------------------------------------------------------------------------
    def _init_state(self):
        sampling = self.engine.inner_model.inner_model.model_sampling
        self.x.copy_(sampling.noise_scaling(self.sigma0, self.noise, self.y))

    def _step(self, i, plan, want_out):
        eng = self.engine
        st = self.sched.steps[i]
        coef = (st.sigma_next - st.sigma) / st.sigma
        last = i + 1 == len(self.sched.steps)
        plan.used = self.draws_before[i]
        out = self.out if (want_out or not self.fused_euler) else None
        if want_out == "each":      # every outer step keeps its own denoised latent
            out = self.outs[i]
        eng._launch_sequence(self.x, self.y, self.noise, self.mask, self._dims, self.tables[i], self.t_model[i],
                             self.sigma[i], self.c, out, self.active[i], plan, False, self.model_options, self.seed,
                             None, self.rng_state.data_ptr(), euler_coef=coef if self.fused_euler else None,
                             skip_prologue=(self.fused_euler and i > 0) or (i == 0 and self.first_replace_noop),
                             next_table=self.tables[i + 1] if (self.fused_euler and not last) else None)
        if not self.fused_euler:
            self.x.add_(self.x - self.out, alpha=coef)

    def _body(self, plan, want_out):
        if not self.external_init:
            self._init_state()
        for i in range(len(self.sched.steps)):
            self._step(i, plan, want_out)

    def _relative_plan(self):
        return self._plan_cls(self.engine.rng, self.x, 1).relative()

    def _capture(self, fn, warm: bool):
        """Capture `fn(plan)` into a CUDA graph.  warm=True first runs it once on a side stream (lazy
        initialisation of whatever the model uses); the node path passes warm=False because the same body has
        already run eagerly as the previous job."""
        eng = self.engine
        counts = (eng.launches, eng.model_calls, eng.substeps_done)
        timer, eng.kernel_timer = eng.kernel_timer, None
        plan = self._relative_plan()   # built BEFORE capture begins: reading the generator's offset is not capturable
        try:
            if warm:
                side = torch.cuda.Stream(device=self.device)
                side.wait_stream(torch.cuda.current_stream(self.device))
                with torch.cuda.stream(side):
                    fn(plan)
                torch.cuda.current_stream(self.device).wait_stream(side)
                eng.launches, eng.model_calls, eng.substeps_done = counts
            graph = torch.cuda.CUDAGraph()
            cap_stream = torch.cuda.Stream(device=self.device)
            cap_stream.wait_stream(torch.cuda.current_stream(self.device))
            with torch.cuda.graph(graph, stream=cap_stream):
                fn(plan)
        finally:
            eng.kernel_timer = timer
        stats = (eng.launches - counts[0], eng.model_calls - counts[1])
        eng.launches, eng.model_calls, eng.substeps_done = counts
        self.captures += 1
        return graph, stats

    def _graph_for(self, key, fn, warm):
        g = self._graphs.get(key)
        if g is None:
            g = self._graphs[key] = self._capture(fn, warm)
        return g

    # ---- one job ---------------------------------------------------------------------------------
    def load_inputs(self, latent_image: torch.Tensor, noise: torch.Tensor, mask, x_init=None):
        """Copies of the request's own inputs into the static buffers (H2D when they are host tensors)."""
        import numpy as np
        from .engine import PackedMask, pack_mask
        self.y.copy_(latent_image, non_blocking=True)
        if noise is None:   # serving hosts that do not need ComfyUI's CPU noise image: draw it on the device
            self.noise.normal_()
        else:
            self.noise.copy_(noise, non_blocking=True)
        if x_init is not None:
            self.x.copy_(x_init, non_blocking=True)
        pm = mask if isinstance(mask, PackedMask) else pack_mask(mask, self.x)
        if self.mask is None or self.mask.data.shape != pm.data.shape or (
                self.mask.row_stride, self.mask.channel_stride) != (pm.row_stride, pm.channel_stride):
            self.mask = PackedMask(torch.empty_like(pm.data), pm.row_stride, pm.channel_stride)
            self._graphs = {}
        self.mask.data.copy_(pm.data, non_blocking=True)
        B = self.shape[0]
        self._dims = _native.Dims(B, self.x.numel() // B, int(np.prod(self.shape[2:])), self.mask.row_stride,
                                  self.mask.channel_stride)

    def run(self, latent_image: torch.Tensor, noise: torch.Tensor, mask, x_out: Optional[torch.Tensor] = None,
            x_init: Optional[torch.Tensor] = None, callback=None, mode: Optional[str] = None, warm: bool = True):
        """callback(i, denoised, x, total_steps) is called on the host after outer step i has been ENQUEUED
        (it sees device tensors in stream order; a callback that only counts steps never synchronises)."""
        import numpy as np
        eng = self.engine
        if self.external_init != (x_init is not None):
            raise ValueError("x_init must be given exactly when the job was built with external_init=True")
        if mode is None:
            mode = "steps" if callback is not None else "job"
        if mode not in ("job", "steps", "eager"):
            raise ValueError(f"unknown mode {mode!r}")
        with torch.cuda.device(self.device):
            before = (eng.launches, eng.model_calls)
            self.load_inputs(latent_image, noise, mask, x_init)
            plan = self._plan_cls(eng.rng, self.x, 1)
            self.rng_state.copy_(torch.from_numpy(plan.state_words().view(np.int64)))
            if self.timing:   # device time of the sampler loop proper: inputs resident, first kernel -> last kernel
                self.last_events = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                self.last_events[0].record()
            n_steps = len(self.sched.steps)
            want_out = callback is not None
            if mode == "job":
                if want_out and self.outs is None:
                    self.outs = [torch.empty_like(self.x) for _ in range(n_steps)]
                each = "each" if want_out else False
                graph, stats = self._graph_for(("job", each), lambda p: self._body(p, each), warm)
                graph.replay()
                eng.launches += stats[0]
                eng.model_calls += stats[1]
                if callback is not None:
                    for i in range(n_steps):
                        callback(i, self.outs[i], self.x, n_steps)
            elif mode == "steps":
                if not self.external_init:
                    self._init_state()
                for i in range(n_steps):
                    graph, stats = self._graph_for(("step", i, want_out), lambda p, i=i: self._step(i, p, want_out), warm)
                    graph.replay()
                    eng.launches += stats[0]
                    eng.model_calls += stats[1]
                    if callback is not None:
                        callback(i, self.out, self.x, n_steps)
            elif mode == "eager":
                rel = self._relative_plan()
                if not self.external_init:
                    self._init_state()
                for i in range(n_steps):
                    self._step(i, rel, want_out)
                    if callback is not None:
                        callback(i, self.out, self.x, n_steps)
            else:
                raise ValueError(f"unknown mode {mode!r}")
            if self.timing:
                self.last_events[1].record()
            plan.consume(self.draws)
            plan.finish()
            eng.substeps_done += self.sched.substeps
            self.launches, self.model_calls = eng.launches - before[0], eng.model_calls - before[1]
            if x_out is not None:
                x_out.copy_(self.x, non_blocking=True)
                return x_out
            return self.x.clone()


class SamplerGraphJob:
    """ANY deterministic k-diffusion sampler around the per-sigma wrapper as ONE CUDA graph per job.

    `runner.GraphedJob` owns the sampler loop, so it only serves Euler.  For the other samplers (heun, dpm_2,
    dpmpp_2m, deis, res_multistep, ...) the loop is third-party Python that calls the wrapper with sigma values only
    it knows.  But for a fixed schedule that sequence is deterministic: the node layer records it during the first,
    eager job of a configuration (`KSamplerX0Inpaint.trace`), this class turns every recorded call into device
    constants (`engine.plan_item`) and then runs the sampler function ITSELF under stream capture -- its Python runs
    once, at capture -- with the wrapper serving the planned calls (`engine.run_planned`: no read-back, no copies).
    The sampler gets the schedule as a CPU tensor so that its own scalar tests (`sigmas[i + 1] == 0`) stay on the host.
    Falls back (exception -> the node layer uses the per-sigma graphs) when the sampler syncs, allocates host
    memory in a way capture forbids, draws its own noise, or calls the model a different number of times.

    Callbacks: the sampler's per-step callback runs at capture time only, so it is recorded there (step index,
    denoised tensor, x tensor -- graph-owned buffers that stay valid) and delivered in order after every replay, the
    same deferred form GraphedJob uses for short jobs."""

    def __init__(self, engine, sampler_function, extra_options, sigmas_cpu: torch.Tensor, trace, shape, device):
        from .engine import _DrawPlan
        self.engine, self.fn, self.extra_options = engine, sampler_function, dict(extra_options or {})
        self.sigmas = sigmas_cpu.detach().to("cpu", torch.float32)
        self.trace = list(trace)            # [(sigma_host [B] CPU tensor, times tuple, n_eff)]
        self.device, self.shape = torch.device(device), tuple(shape)
        mk = lambda: torch.empty(self.shape, dtype=torch.float32, device=self.device)
        self.x0, self.y, self.noise, self.c = mk(), mk(), mk(), mk()
        self.mask = None
        self.rng_state = torch.zeros(2, dtype=torch.int64, device=self.device)
        self.items = None
        self.graph = None
        self.result = None
        self.recorded = []                  # callbacks seen at capture: (i, denoised, x)
        self.draws = 0
        self.launches = self.model_calls = self.substeps = 0
        self.captures = 0
        self._plan_cls = _DrawPlan
        self.timing, self.last_events = False, None

    def _load(self, latent_image, noise, pm, x_init):
        import numpy as np
        from .engine import PackedMask
        self.y.copy_(latent_image, non_blocking=True)
        self.noise.copy_(noise, non_blocking=True)
        self.x0.copy_(x_init, non_blocking=True)
        if self.mask is None or self.mask.data.shape != pm.data.shape or (
                self.mask.row_stride, self.mask.channel_stride) != (pm.row_stride, pm.channel_stride):
            self.mask = PackedMask(torch.empty_like(pm.data), pm.row_stride, pm.channel_stride)
            self.graph = None
        self.mask.data.copy_(pm.data, non_blocking=True)
        B = self.shape[0]
        self.dims = _native.Dims(B, self.x0.numel() // B, int(np.prod(self.shape[2:])), self.mask.row_stride,
                                 self.mask.channel_stride)

    def _capture(self, model_k, extra_args, want_callbacks):
        eng = self.engine
        B = self.shape[0]
        self.items = []
        for sigma_host, times, n_eff in self.trace:
            item = eng.plan_item(B, sigma_host, times, n_eff, self.device)
            if item is None:
                raise RuntimeError("noise_scaling is not a linear form")
            self.items.append(item)
        plan = self._plan_cls(eng.rng, self.x0, 1).relative()   # before capture: reads the generator once
        counts = (eng.launches, eng.model_calls, eng.substeps_done)
        state = {"pos": 0}
        job = self

        def planned(x, model_options, seed):
            if state["pos"] >= len(job.items):
                raise RuntimeError("the sampler called the model more often than in its recorded job")
            item = job.items[state["pos"]]
            state["pos"] += 1
            return eng.run_planned(x, item, job.y, job.noise, job.mask, job.dims, job.c, plan, job.rng_state.data_ptr(),
                                   model_options, seed)
        model_k.planned_call = planned
        self.recorded = []
        k_callback = None
        if want_callbacks:
            k_callback = lambda d: job.recorded.append((d["i"], d["denoised"], d["x"]))  # noqa: E731
        graph = torch.cuda.CUDAGraph()
        cap_stream = torch.cuda.Stream(device=self.device)
        cap_stream.wait_stream(torch.cuda.current_stream(self.device))
        try:
            with torch.cuda.graph(graph, stream=cap_stream):
                self.result = self.fn(model_k, self.x0, self.sigmas, extra_args=extra_args, callback=k_callback,
                                      disable=True, **self.extra_options)
        finally:
            model_k.planned_call = None
        if state["pos"] != len(self.items):
            raise RuntimeError("the sampler called the model less often than in its recorded job")
        self.graph, self.draws = graph, plan.used
        self.launches, self.model_calls = eng.launches - counts[0], eng.model_calls - counts[1]
        self.substeps = eng.substeps_done - counts[2]
        eng.launches, eng.model_calls, eng.substeps_done = counts
        self.captures += 1

    def run(self, model_k, extra_args, latent_image, noise, pm, x_init, callback=None):
        """callback(i, denoised, x, total_steps): ComfyUI's; delivered after the replay, in the sampler's order."""
        import numpy as np
        eng = self.engine
        with torch.cuda.device(self.device):
            self._load(latent_image, noise, pm, x_init)
            if self.graph is None:
                self._capture(model_k, extra_args, callback is not None)
            plan = self._plan_cls(eng.rng, self.x0, 1)
            self.rng_state.copy_(torch.from_numpy(plan.state_words().view(np.int64)))
            if self.timing:
                self.last_events = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                self.last_events[0].record()
            self.graph.replay()
            if self.timing:
                self.last_events[1].record()
            plan.consume(self.draws)
            plan.finish()
            eng.launches += self.launches
            eng.model_calls += self.model_calls
            eng.substeps_done += self.substeps
            if callback is not None:
                total = len(self.sigmas) - 1
                for i, den, xx in self.recorded:
                    callback(i, den, xx, total)
            return self.result.clone()
