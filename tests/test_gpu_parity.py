"""GPU parity: the CUDA path (through the C ABI) against the reference's own
outputs (golden fixtures) and against the oracle on identical inputs.

Tolerances.  BASELINE.json's bar is 1e-3 relative fp32 on the final latent.
The kernels agree with the reference to fp32 round-off, so the tests assert a
much tighter engineering bound (TIGHT) and keep the contractual bound as a
named constant for the record.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import golden_names, load_golden
from _support import make_model, max_rel, rel_l2, synth_inputs
from oracle import langevin_oracle as O

pytestmark = pytest.mark.gpu

CONTRACT = 1e-3  # north_star tolerance
TIGHT = 2e-5     # what fp32 round-off between two orderings of the same math allows


def _engine(model, meta=None, **kw):
    from lanpaint_b200.engine import LanPaint
    meta = meta or {}
    return LanPaint(model, NSteps=meta.get("n_steps", 5), Friction=meta.get("friction", 15.0),
                    Lambda=meta.get("lam", 5.0), Beta=meta.get("beta", 1.0), StepSize=meta.get("step_size", 0.2),
                    IS_FLUX=False, IS_FLOW=meta.get("flow", False), MinStepFrac=meta.get("min_step_frac", 1.0), **kw)


def _hyper(meta):
    return O.Hyper(n_steps=meta["n_steps"], lam=meta["lam"], beta=meta["beta"], step_size=meta["step_size"],
                   min_step_frac=meta["min_step_frac"], flow=meta["flow"])


# ----------------------------------------------------------------------------
# 1. against the reference's own outputs (fixtures generated from /root/reference)
# ----------------------------------------------------------------------------
@pytest.mark.parametrize("name", golden_names())
def test_engine_matches_reference_golden(name, cuda_device):
    from lanpaint_b200.engine import NoiseTape
    g = load_golden(name)
    meta = g["meta"]
    dev = cuda_device
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    x, y, noise, mask = t(g["x"]), t(g["y"]), t(g["noise"]), t(g["mask_full"])
    sigma = t(g["sigma"])
    times = (t(g["ve"]), t(g["abt"]), t(g["flow_t"]))
    tape = NoiseTape([t(d) for d in g["tape"]])
    model = make_model(meta["model"], meta["flow"])
    eng = _engine(model, meta, rng=tape)
    out = eng(x, y, noise, sigma, mask, times, {}, 0, n_steps=meta["n_steps"])
    torch.cuda.synchronize()
    assert tape.pos == meta["n_draws"], "draw count/order differs from the reference"
    e_out = max_rel(out, torch.from_numpy(g["out"]))
    e_x = max_rel(x, torch.from_numpy(g["x_new"]))  # x is rewritten in place (lanpaint.py:156)
    assert e_out <= TIGHT and e_x <= TIGHT, (name, e_out, e_x)
    assert max(e_out, e_x) <= CONTRACT
    assert model.calls == meta["n_steps"] + 1


# ----------------------------------------------------------------------------
# 2. same seed on the GPU: torch's global CUDA generator, reference draw order
# ----------------------------------------------------------------------------
@pytest.mark.parametrize("shape,flow,n,sigma", [
    ((1, 4, 64, 64), False, 5, [2.0]),          # BASELINE config 1
    ((1, 4, 128, 128), False, 5, [7.0]),        # config 2 shape
    ((2, 4, 32, 32), False, 3, [1.0, 1.0]),     # batch -> flow-form replace quirk
    ((1, 16, 32, 32), True, 4, [0.6]),          # flow
    ((1, 16, 21, 80, 45), True, 2, [0.8]),      # Wan-sized 5-D latent: > one torch randn wave
    ((1, 3, 5, 7), False, 3, [1.5]),            # odd sizes -> scalar path
])
def test_same_seed_matches_oracle_on_gpu(shape, flow, n, sigma, cuda_device):
    dev = cuda_device
    x, y, noise, m = synth_inputs(shape, seed=3, device=dev)
    mask = m.expand(shape).contiguous()
    sig = torch.tensor(sigma, device=dev)
    times = O.times_from_sigma(sig, flow)
    hp = O.Hyper(n_steps=n, min_step_frac=1.0, flow=flow)
    torch.manual_seed(1234)
    out_o, x_o = O.outer_step(make_model("two_heads", flow), x.clone(), y, noise, sig, mask, times, hp, n_steps=n)
    off_o = torch.cuda.default_generators[dev.index].get_offset()

    torch.manual_seed(1234)
    eng = _engine(make_model("two_heads", flow), dict(n_steps=n, flow=flow), rng="torch")
    xe = x.clone()
    out_e = eng(xe, y, noise, sig, mask, tuple(times), {}, 0, n_steps=n)
    off_e = torch.cuda.default_generators[dev.index].get_offset()
    assert off_e == off_o, "generator must advance exactly as the reference's randn_like calls do"
    assert max_rel(out_e, out_o) <= TIGHT and max_rel(xe, x_o) <= TIGHT, (max_rel(out_e, out_o), max_rel(xe, x_o))


@pytest.mark.parametrize("n", [1, 255, 256, 4097, 303104, 303105, 1209600, 2097152 + 3])
def test_torch_stream_is_bit_exact(n, cuda_device):
    """lp_fill_normal_f32(LP_RNG_TORCH) == torch.randn on the same (seed, offset)."""
    from lanpaint_b200 import _native
    lib = _native.load()
    dev = cuda_device
    gen = torch.cuda.default_generators[dev.index]
    torch.manual_seed(77)
    _ = torch.randn(5, device=dev)  # move the offset off zero
    seed, off = gen.initial_seed(), gen.get_offset()
    ref = torch.randn(n, device=dev)
    out = torch.empty(n, device=dev)
    r = _native.Rng(mode=_native.RNG_TORCH, seed=seed, draw0=off)
    rc = lib.lp_fill_normal_f32(C.c_void_p(out.data_ptr()), n, C.byref(r),
                                C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0
    g, inc = C.c_int64(0), C.c_uint64(0)
    assert lib.lp_torch_randn_geometry(n, dev.index, C.byref(g), C.byref(inc)) == 0
    assert gen.get_offset() - off == inc.value
    same = torch.equal(out, ref)
    if not same:  # a libdevice logf difference between toolkits would show up here as 1-ulp noise
        assert (out - ref).abs().max().item() <= 1e-6, (out - ref).abs().max().item()
    assert same


def test_philox_stream_statistics_and_determinism(cuda_device):
    from lanpaint_b200 import _native
    lib = _native.load()
    dev = cuda_device
    n = 1 << 22
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    a, b, c = (torch.empty(n, device=dev) for _ in range(3))
    for buf, draw in ((a, 0), (b, 1), (c, 0)):
        r = _native.Rng(mode=_native.RNG_PHILOX, seed=99, draw0=draw)
        assert lib.lp_fill_normal_f32(C.c_void_p(buf.data_ptr()), n, C.byref(r), s) == 0
    assert torch.equal(a, c)
    assert abs(a.mean().item()) < 3e-3 and abs(a.var().item() - 1.0) < 5e-3
    assert abs((a * b).mean().item()) < 3e-3          # draws are independent
    assert abs((a[1:] * a[:-1]).mean().item()) < 3e-3  # neighbours are independent
    assert abs((a ** 4).mean().item() - 3.0) < 0.05    # Gaussian kurtosis
    assert a.abs().max().item() < 7.0


# ----------------------------------------------------------------------------
# 3. BASELINE sizes: direct parity against the oracle run on the GPU + properties
# ----------------------------------------------------------------------------
@pytest.mark.parametrize("shape,flow,n", [
    ((8, 4, 128, 128), False, 5),      # north_star "batch 8" target shape
    ((32, 4, 128, 128), False, 10),    # config 3 unsharded
    ((1, 16, 128, 128), True, 5),      # config 4 at the ComfyUI boundary
    ((1, 16, 21, 80, 45), True, 5),    # config 5
])
def test_full_size_tape_parity_and_properties(shape, flow, n, cuda_device):
    from lanpaint_b200.engine import NoiseTape
    dev = cuda_device
    x, y, noise, m = synth_inputs(shape, seed=11, device=dev)
    mask = m.expand(shape).contiguous()
    B = shape[0]
    sig = torch.full((B,), 0.7 if flow else 2.5, device=dev)
    times = O.times_from_sigma(sig, flow)
    hp = O.Hyper(n_steps=n, min_step_frac=1.0, flow=flow)
    tape = O.NoiseTape(generator=torch.Generator().manual_seed(5))
    out_o, x_o = O.outer_step(make_model("two_heads", flow), x.clone(), y, noise, sig, mask, times, hp,
                              n_steps=n, draw=tape)
    eng = _engine(make_model("two_heads", flow), dict(n_steps=n, flow=flow), rng=NoiseTape(tape.recorded))
    xe = x.clone()
    out_e = eng(xe, y, noise, sig, m, tuple(times), {}, 0, n_steps=n)  # [B,1,...] mask: 1/C byte per element path
    assert max_rel(out_e, out_o) <= TIGHT and max_rel(xe, x_o) <= TIGHT
    assert rel_l2(xe, x_o) <= 1e-6
    # property: the known region of `out` is exactly the clean latent (lanpaint.py:154)
    known = mask.bool()
    assert torch.equal(out_e[known], y[known])
    # property: one launch per sub-step (+ mask pack, prologue, epilogue)
    assert eng.launches == n + 3 and eng.model_calls == n + 1


def test_batch_equals_independent_requests(cuda_device):
    """Samples never interact: a batch run == each sample run alone (per_sample replace)."""
    from lanpaint_b200.engine import NoiseTape
    dev = cuda_device
    shape = (4, 4, 32, 32)
    x, y, noise, m = synth_inputs(shape, seed=5, device=dev)
    sig = torch.tensor([0.5, 2.0, 6.0, 13.0], device=dev)
    times = O.times_from_sigma(sig, False)
    draws = [torch.randn(shape, device=dev) for _ in range(5)]
    eng = _engine(make_model("two_heads", False), dict(n_steps=3), rng=NoiseTape(draws), batched_replace="per_sample")
    xb = x.clone()
    out_b = eng(xb, y, noise, sig, m, tuple(times), {}, 0, n_steps=3)
    for b in range(4):
        sl = slice(b, b + 1)
        e1 = _engine(make_model("two_heads", False), dict(n_steps=3), rng=NoiseTape([d[sl].contiguous() for d in draws]))
        x1 = x[sl].clone()
        o1 = e1(x1, y[sl].contiguous(), noise[sl].contiguous(), sig[sl], m[sl].contiguous(),
                tuple(t[sl] for t in times), {}, 0, n_steps=3)
        assert torch.equal(o1, out_b[sl]) and torch.equal(x1, xb[sl])


def test_vector_and_scalar_paths_agree_bitwise(cuda_device):
    """A 4-byte-misaligned view forces the scalar kernels; results must equal the 128-bit path."""
    from lanpaint_b200.engine import NoiseTape
    dev = cuda_device
    shape = (2, 4, 16, 16)
    x, y, noise, m = synth_inputs(shape, seed=9, device=dev)
    sig = torch.tensor([1.5, 1.5], device=dev)
    times = O.times_from_sigma(sig, False)
    draws = [torch.randn(shape, device=dev) for _ in range(5)]

    def run(xin):
        eng = _engine(make_model("two_heads", False), dict(n_steps=3), rng=NoiseTape(draws))
        out = eng(xin, y, noise, sig, m, tuple(times), {}, 0, n_steps=3)
        return out, xin

    o_vec, x_vec = run(x.clone())
    pad = torch.empty(x.numel() + 1, device=dev)
    x_mis = pad[1:].view(shape)
    x_mis.copy_(x)
    assert x_mis.data_ptr() % 16 != 0
    o_sc, x_sc = run(x_mis)
    assert torch.equal(o_vec, o_sc) and torch.equal(x_vec, x_sc)


def test_philox_mode_reproducible_and_sane(cuda_device):
    dev = cuda_device
    shape = (2, 4, 64, 64)
    x, y, noise, m = synth_inputs(shape, seed=2, device=dev)
    sig = torch.tensor([2.0, 2.0], device=dev)
    times = O.times_from_sigma(sig, False)

    def run(seed):
        torch.manual_seed(seed)
        eng = _engine(make_model("two_heads", False), dict(n_steps=4), rng="philox")
        xx = x.clone()
        return eng(xx, y, noise, sig, m, tuple(times), {}, 0, n_steps=4), xx

    o1, x1 = run(1)
    o2, x2 = run(1)
    o3, x3 = run(2)
    assert torch.equal(x1, x2) and torch.equal(o1, o2)
    assert not torch.equal(x1, x3)
    # distributional sanity against the oracle with its own (different) stream
    torch.manual_seed(1)
    _, x_o = O.outer_step(make_model("two_heads", False), x.clone(), y, noise, sig, m.expand(shape), times,
                          O.Hyper(n_steps=4, min_step_frac=1.0), n_steps=4)
    free = ~m.expand(shape).bool()
    assert abs(x1[free].std().item() / x_o[free].std().item() - 1.0) < 0.05
    assert abs(x1[free].mean().item() - x_o[free].mean().item()) < 0.1


# ----------------------------------------------------------------------------
# 4. edge cases and error behaviour
# ----------------------------------------------------------------------------
def test_empty_batch_is_a_no_op(cuda_device):
    dev = cuda_device
    x = torch.empty(0, 4, 16, 16, device=dev)
    model = make_model("two_heads", False)
    eng = _engine(model, dict(n_steps=3))
    e = torch.empty(0, device=dev)
    out = eng(x, x, x, e, x, (e, e, e), {}, 0, n_steps=3)
    assert out.shape == x.shape and model.calls == 0


def test_cpu_tensor_is_rejected_loudly():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    eng = _engine(make_model("identity", False))
    x = torch.zeros(1, 4, 8, 8)
    with pytest.raises(RuntimeError):
        eng(x, x, x, torch.tensor([1.0]), x, (torch.tensor([1.0]),) * 3, {}, 0)


def test_empty_model_output_raises_value_error(cuda_device):
    class Empty(O.PointwiseDenoiser):
        def __call__(self, x, sigma, model_options=None, seed=None):
            return ()
    dev = cuda_device
    x, y, noise, m = synth_inputs((1, 4, 8, 8), device=dev)
    sig = torch.tensor([1.0], device=dev)
    eng = _engine(Empty(O.VESampling()))
    with pytest.raises(ValueError, match="Model output is empty"):
        eng(x, y, noise, sig, m, tuple(O.times_from_sigma(sig, False)), {}, 0, n_steps=2)


def test_noncontiguous_and_half_inputs(cuda_device):
    from lanpaint_b200.engine import NoiseTape
    dev = cuda_device
    shape = (1, 4, 16, 16)
    x, y, noise, m = synth_inputs(shape, seed=4, device=dev)
    sig = torch.tensor([2.0], device=dev)
    times = O.times_from_sigma(sig, False)
    draws = [torch.randn(shape, device=dev) for _ in range(3)]
    ref_eng = _engine(make_model("two_heads", False), dict(n_steps=2), rng=NoiseTape(draws))
    x_ref = x.clone()
    o_ref = ref_eng(x_ref, y, noise, sig, m, tuple(times), {}, 0, n_steps=2)
    # channels-last strided x: the in-place contract must still hold
    x_nc = x.clone().permute(0, 2, 3, 1).contiguous().permute(0, 3, 1, 2)
    assert not x_nc.is_contiguous()
    eng = _engine(make_model("two_heads", False), dict(n_steps=2), rng=NoiseTape(draws))
    o = eng(x_nc, y, noise, sig, m, tuple(times), {}, 0, n_steps=2)
    assert torch.equal(o, o_ref) and torch.equal(x_nc, x_ref)


def test_flat_3d_latent_and_zero_steps(cuda_device):
    """[1,1,8] flat pack, n_steps=0: replace + final call only (tests/test_av_schedule.py:204-219 shape)."""
    dev = cuda_device
    x = torch.zeros(1, 1, 8, device=dev)
    y = torch.zeros_like(x)
    noise = torch.ones_like(x)
    sig = torch.tensor([0.5], device=dev)
    mask = torch.ones_like(x)
    model = make_model("identity", True)
    eng = _engine(model, dict(n_steps=0, flow=True, lam=1.0))
    eng(x, y, noise, sig, mask, (torch.tensor([1.0], device=dev), torch.tensor([0.5], device=dev), sig), None, 0,
        n_steps=0)
    assert torch.allclose(model.last_input.flatten(), torch.full((8,), 0.5, device=dev))
    assert model.calls == 1


def test_c_abi_rejects_bad_arguments():
    from lanpaint_b200 import _native
    lib = _native.load()
    d = _native.Dims(1, 16, 16, 16, 0)
    r = _native.Rng(mode=_native.RNG_PHILOX)
    assert lib.lp_substep_f32(None, None, None, None, None, None, None, None, None, C.byref(d), C.byref(r), 1, None) == 1
    assert lib.lp_prologue_f32(None, None, None, None, None, None, None, C.byref(d), None) == 1
    assert lib.lp_status_string(1).decode() == "invalid argument"


def test_advance_abi_matches_oracle(cuda_device):
    """lp_advance_f32 == advance_time_overdamped (lanpaint.py:232-254) on the model-space state."""
    from lanpaint_b200 import _native
    from lanpaint_b200.schedule import Hyper, build_table
    lib = _native.load()
    dev = cuda_device
    B, Cc, S = 2, 4, 64
    torch.manual_seed(0)
    x = torch.randn(B, Cc, S, device=dev)
    c = torch.randn_like(x)
    xi = torch.randn_like(x)
    mask = (torch.rand(B, 1, S, device=dev) < 0.5)
    sig = torch.tensor([0.7, 3.0], device=dev)
    ve, abt, _ = O.times_from_sigma(sig, False)
    hp = Hyper(0.2, 5.0, 1.0, 1.0, False)
    tab = torch.from_numpy(build_table(abt.cpu().numpy(), ve.cpu().numpy(), hp)).to(dev)
    for half in (0, 1):
        xk = x.clone()
        d = _native.Dims(B, Cc * S, S, S, 0)
        r = _native.Rng(mode=_native.RNG_TAPE, tape0=xi.data_ptr())
        m8 = mask.to(torch.uint8).contiguous()
        rc = lib.lp_advance_f32(C.c_void_p(xk.data_ptr()), C.c_void_p(c.data_ptr()), C.c_void_p(m8.data_ptr()),
                                C.c_void_p(tab.data_ptr()), C.byref(d), C.byref(r), half,
                                C.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == 0
        # oracle in VP space, fp64
        mf = mask.expand(B, Cc, S).double()
        abt_b = abt.double().view(B, 1, 1)
        Sx = (1 + ve.double() ** 2).sqrt().view(B, 1, 1)
        step = 0.2 * (1 - abt_b).clamp(min=1.0)
        cf = O.branch_coefficients(abt_b, step, torch.ones_like(abt_b), torch.ones_like(abt_b), 5.0)
        A = cf.A_x * (1 - mf) + cf.A_y * mf
        D = cf.D_x * (1 - mf) + cf.D_y * mf
        dt = cf.half_dt_x * (1 - mf) + cf.half_dt_y * mf
        h = dt / 2 if half else dt
        want = O.ou_advance(x.double() / Sx, h, A, c.double(), D, lambda t: xi.double()) * Sx
        assert max_rel(xk, want) <= TIGHT


def test_synth_denoiser_kernel_matches_torch(cuda_device):
    from lanpaint_b200 import _native
    lib = _native.load()
    dev = cuda_device
    x = torch.randn(3, 4, 33, 31, device=dev)
    h0, h1 = torch.empty_like(x), torch.empty_like(x)
    coef = (C.c_float * 5)(0.7, 0.1, 0.0, 0.6, -0.05)
    rc = lib.lp_synth_denoiser_f32(C.c_void_p(x.data_ptr()), C.c_void_p(h0.data_ptr()), C.c_void_p(h1.data_ptr()),
                                   x.numel(), coef, C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0
    w0, w1 = make_model("two_heads", False)(x, None)
    assert max_rel(h0, w0) <= 1e-6 and max_rel(h1, w1) <= 1e-6


# ----------------------------------------------------------------------------
# 5. CUDA-graph replay of whole outer steps
# ----------------------------------------------------------------------------
@pytest.mark.parametrize("rng", ["philox", "torch"])
def test_graph_replay_equals_eager_launches(rng, cuda_device):
    from lanpaint_b200.runner import SynthDenoiser, VESampling
    dev = cuda_device
    shape = (4, 4, 64, 64)
    x, y, noise, m = synth_inputs(shape, seed=21, device=dev)
    res = {}
    for mode in (False, True):
        torch.manual_seed(9)
        eng = _engine(SynthDenoiser(VESampling()), dict(n_steps=5), rng=rng, cuda_graph=mode,
                      batched_replace="per_sample")
        outs = []
        xx = x.clone()
        for sig_v, n in ((9.0, 5), (3.0, 5), (1.0, 3), (0.2, 0)):   # two sigmas share the n=5 graph
            sig = torch.full((4,), sig_v)                              # CPU-resident: the sync-free path
            times = O.times_from_sigma(sig, False)
            outs.append(eng(xx, y, noise, sig, m, tuple(times), None, 0, n_steps=n).clone())
        res[mode] = (outs, xx.clone(), eng, torch.cuda.default_generators[dev.index].get_offset())
    for a, b in zip(res[False][0], res[True][0]):
        assert torch.equal(a, b)
    assert torch.equal(res[False][1], res[True][1])
    assert res[False][3] == res[True][3]                  # generator advanced identically
    g = res[True][2]
    assert len([v for v in g._graphs.values() if v]) == 3  # n = 5, 3, 0 -> three graphs, sigma is data
    assert g.launches == res[False][2].launches and g.model_calls == res[False][2].model_calls


def test_graph_capture_failure_falls_back_to_eager(cuda_device):
    class Syncing(O.PointwiseDenoiser):
        def __call__(self, x, sigma, model_options=None, seed=None):
            float(x.sum())  # a host sync: illegal under stream capture
            return super().__call__(x, sigma)
    dev = cuda_device
    shape = (1, 4, 16, 16)
    x, y, noise, m = synth_inputs(shape, seed=2, device=dev)
    sig = torch.tensor([2.0])
    times = O.times_from_sigma(sig, False)
    torch.manual_seed(3)
    eng = _engine(Syncing(O.VESampling()), dict(n_steps=2), rng="philox", cuda_graph=True)
    with pytest.warns(UserWarning, match="capture failed"):
        out = eng(x.clone(), y, noise, sig, m, tuple(times), None, 0, n_steps=2)
    torch.manual_seed(3)
    ref = _engine(O.PointwiseDenoiser(O.VESampling()), dict(n_steps=2), rng="philox")
    assert torch.equal(out, ref(x.clone(), y, noise, sig, m, tuple(times), None, 0, n_steps=2))
    # the aborted capture must not leave torch's generator unusable
    assert torch.isfinite(torch.rand(8, device=dev)).all() and torch.isfinite(torch.randn(8, device=dev)).all()


# ----------------------------------------------------------------------------
# 6. merged Gaussian kick (LP_SUBSTEP_MERGE_NOISE, philox stream only)
# ----------------------------------------------------------------------------
def _raw_substep(lib, x, x0, x0b, y, m8, c, tab, dims, flags, seed=5, draw=0):
    from lanpaint_b200 import _native
    P = C.c_void_p
    r = _native.Rng(mode=_native.RNG_PHILOX, seed=seed, draw0=draw, draw1=draw + 1)
    rc = lib.lp_substep_f32(P(x.data_ptr()), P(x0.data_ptr()), P(x0b.data_ptr()), P(y.data_ptr()), P(m8.data_ptr()),
                            P(c.data_ptr()), None, None, P(tab.data_ptr()), C.byref(dims), C.byref(r), flags,
                            P(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, rc


@pytest.mark.parametrize("first", [0, 1])
def test_merged_noise_same_drift_and_same_variance(first, cuda_device):
    from lanpaint_b200 import _native
    from lanpaint_b200.schedule import Hyper, build_table
    lib = _native.load()
    dev = cuda_device
    B, Cc, S = 2, 4, 1 << 16
    sig = torch.tensor([0.8, 4.0])
    ve, abt, _ = O.times_from_sigma(sig, False)
    tab_np = build_table(abt.numpy(), ve.numpy(), Hyper(0.2, 5.0, 1.0, 1.0, False))
    dims = _native.Dims(B, Cc * S, S, S, 0)
    m8 = (torch.rand(B, 1, S, device=dev) < 0.5).to(torch.uint8)
    base = [torch.randn(B, Cc, S, device=dev) for _ in range(5)]
    F2, FM = 2 | first, 2 | 8 | first

    # (a) with every kick std zeroed, the merged and the two-draw kernels are the same arithmetic
    quiet = tab_np.copy()
    quiet[:, [8 + 4, 8 + 7, 16 + 4, 16 + 7, 24, 25, 26, 27]] = 0.0
    tq = torch.from_numpy(quiet).to(dev)
    outs = []
    for flags in (F2, FM):
        x, x0, x0b, y, c = (t.clone() for t in base)
        _raw_substep(lib, x, x0, x0b, y, m8, c, tq, dims, flags)
        outs.append((x, c))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])

    # (b) with constant operands the output is (constant + kick): its per-class variance must agree
    tab = torch.from_numpy(tab_np).to(dev)
    res = []
    for flags in (F2, FM):
        x, x0, x0b, y, c = (torch.full((B, Cc, S), v, device=dev) for v in (0.3, -0.2, 0.5, 0.1, 0.05))
        _raw_substep(lib, x, x0, x0b, y, m8, c, tab, dims, flags)
        res.append(x)
    known = m8.bool().expand(B, Cc, S)
    for b in range(B):
        for cls in (known[b], ~known[b]):
            v2, vm = res[0][b][cls].var().item(), res[1][b][cls].var().item()
            m2, mm = res[0][b][cls].mean().item(), res[1][b][cls].mean().item()
            assert abs(vm / v2 - 1.0) < 0.03, (b, v2, vm)
            assert abs(mm - m2) < 4.0 * (v2 / cls.sum().item()) ** 0.5 + 1e-4
    # the ABI refuses the flag where it would break stream parity
    x, x0, x0b, y, c = (t.clone() for t in base)
    P = C.c_void_p
    r = _native.Rng(mode=_native.RNG_TORCH, seed=1, draw0=0, draw1=4)
    assert lib.lp_substep_f32(P(x.data_ptr()), P(x0.data_ptr()), P(x0b.data_ptr()), P(y.data_ptr()), P(m8.data_ptr()),
                              P(c.data_ptr()), None, None, P(tab.data_ptr()), C.byref(dims), C.byref(r), FM, None) == 1


@pytest.mark.parametrize("rng", ["philox", "torch"])
def test_whole_job_graph_equals_step_by_step(rng, cuda_device):
    """runner.GraphedJob (one CUDA graph for the 20-step job) == euler_inpaint with eager launches."""
    from lanpaint_b200.runner import GraphedJob, HostSchedule, SynthDenoiser, VESampling, euler_inpaint, karras_sigmas
    dev = cuda_device
    shape = (3, 4, 32, 32)
    _, y, noise, m = synth_inputs(shape, seed=8, device=dev)
    sched = HostSchedule(karras_sigmas(20), 3, 5)
    assert sched.substeps == 53 and sched.model_calls == 73

    def engine():
        return _engine(SynthDenoiser(VESampling()), dict(n_steps=5), rng=rng, batched_replace="per_sample")

    torch.manual_seed(4)
    e1 = engine()
    want = euler_inpaint(e1, y, noise, m, sched)
    off1 = torch.cuda.default_generators[dev.index].get_offset()
    torch.manual_seed(4)
    e2 = engine()
    job = GraphedJob(e2, sched, shape, dev, fused_euler=False)
    got = job.run(y, noise, m)
    off2 = torch.cuda.default_generators[dev.index].get_offset()
    assert torch.equal(got, want) and off1 == off2
    torch.manual_seed(4)
    fused = GraphedJob(engine(), sched, shape, dev, fused_euler=True).run(y, noise, m)   # Euler inside the epilogue
    assert max_rel(fused, want) <= 1e-5
    assert e2.model_calls == e1.model_calls == 73 and e2.substeps_done == 53
    again = job.run(y, noise, m)          # a second request batch: fresh noise, same graph
    assert not torch.equal(again, got) and torch.isfinite(again).all()


# ----------------------------------------------------------------------------
# 7. the reference's lower-level entry point: langevin_dynamics(x_t, score, ...)
# ----------------------------------------------------------------------------
def test_langevin_dynamics_method_matches_oracle(cuda_device):
    """Same call as the reference's tests/test_sho_regression.py, checked numerically against the oracle's
    restatement of lanpaint.py:192-293 for a first and a steady sub-step with an arbitrary score callback."""
    from lanpaint_b200.engine import NoiseTape
    from lanpaint_b200.state import LangevinState
    dev = cuda_device
    torch.manual_seed(0)
    shape = (2, 4, 16, 16)
    x = torch.randn(shape, device=dev)
    mask = (torch.rand(2, 1, 16, 16, device=dev) < 0.5).float().expand(shape).contiguous()
    score = lambda z: -0.3 * z + 0.1 * torch.tanh(z)
    abt = torch.tensor([0.5, 0.8], device=dev)
    times = (torch.tensor([1.0, 0.5], device=dev), abt, torch.tensor([0.5, 0.3], device=dev))
    step = torch.tensor([0.1, 0.04], device=dev).view(2, 1, 1, 1)
    draws = [torch.randn(shape, device=dev) for _ in range(3)]
    hp = O.Hyper(n_steps=10, friction=1.0, lam=2.0, beta=1.0, step_size=0.1)
    ones = torch.ones(2, 1, 1, 1, device=dev)
    tape_o = O.NoiseTape(draws)
    x1_o, st1_o = O.langevin_substep(x, score, mask, step, O.Times(*times), hp, None, tape_o, ones, 1.5 * ones)
    x2_o, st2_o = O.langevin_substep(x1_o, score, mask, step, O.Times(*times), hp, st1_o, tape_o, ones, 1.5 * ones)

    eng = _engine(make_model("identity", False), dict(lam=2.0, step_size=0.1), rng=NoiseTape(draws))
    eng.img_dim_size = 4
    x1, st1 = eng.langevin_dynamics(x, score, mask, step, times, sigma_x=ones, sigma_y=1.5 * ones)
    assert isinstance(st1, LangevinState) and st1.v is None and st1[1] is st1.C and st1[2] is st1.x0
    x2, st2 = eng.langevin_dynamics(x1, score, mask, step, times, sigma_x=ones, sigma_y=1.5 * ones, args=st1)
    for got, want in ((x1, x1_o), (st1.C, st1_o.C), (st1.x0, st1_o.x0), (x2, x2_o), (st2.C, st2_o.C), (st2.x0, st2_o.x0)):
        assert max_rel(got, want) <= TIGHT
    assert torch.isfinite(x2).all()
    # zero step size: untouched state, like lanpaint.py:205
    x3, st3 = eng.langevin_dynamics(x, score, mask, 0 * step, times, sigma_x=ones, sigma_y=ones)
    assert x3 is x and st3 is None


def test_graph_capture_of_a_torch_module_denoiser(cuda_device):
    """The model call stays ordinary PyTorch code (here a small conv net with two heads and a sigma
    embedding); the engine captures it together with its own kernels and replays the graph."""
    dev = cuda_device

    class TinyNet(torch.nn.Module):
        def __init__(self):
            super().__init__()
            g = torch.Generator().manual_seed(0)
            self.c1 = torch.nn.Conv2d(4, 32, 3, padding=1)
            self.c2 = torch.nn.Conv2d(32, 8, 3, padding=1)
            for p in self.parameters():
                p.data = torch.randn(p.shape, generator=g) * 0.05

        def forward(self, x, sigma, model_options=None, seed=None):
            emb = (1.0 / (1.0 + sigma ** 2)).view(-1, 1, 1, 1)
            h = torch.nn.functional.silu(self.c1(x * emb))
            o = self.c2(h)
            return x * emb + o[:, :4], x * emb + o[:, 4:]

    class Guider:   # the engine-seam protocol around the module (what ComfyUI's CFGGuider is)
        def __init__(self, module):
            self.module = module
            self.inner_model = self
            self.model_sampling = O.VESampling()

        def __call__(self, x, sigma, model_options=None, seed=None):
            return self.module(x, sigma)

    net = Guider(TinyNet().to(dev).eval())
    shape = (2, 4, 32, 32)
    x, y, noise, m = synth_inputs(shape, seed=13, device=dev)
    res = {}
    with torch.no_grad():
        for mode in (False, True):
            torch.manual_seed(21)
            eng = _engine(net, dict(n_steps=3), rng="philox", cuda_graph=mode, batched_replace="per_sample")
            xx = x.clone()
            outs = []
            for sv in (5.0, 1.5):
                sig = torch.full((2,), sv)
                outs.append(eng(xx, y, noise, sig, m, tuple(O.times_from_sigma(sig, False)), None, 0, n_steps=3))
            res[mode] = (outs, xx, eng)
    assert len([g for g in res[True][2]._graphs.values() if g]) == 1
    for a, b in zip(res[False][0], res[True][0]):
        assert max_rel(a, b) <= 1e-5
    assert max_rel(res[False][1], res[True][1]) <= 1e-5


# ----------------------------------------------------------------------------
# 8. randomized configurations (seeded): shapes, mask layouts, head aliasing, schedules, hyper-parameters
# ----------------------------------------------------------------------------
def _random_cases(n, seed=20260922):
    rng = np.random.default_rng(seed)
    cases = []
    for k in range(n):
        ndim = int(rng.choice([3, 4, 4, 4, 5]))
        B = int(rng.choice([1, 1, 2, 3]))
        Cc = int(rng.choice([1, 3, 4, 16]))
        sp = tuple(int(v) for v in rng.choice([2, 3, 4, 5, 8, 12, 16], size=ndim - 2))
        flow = bool(rng.random() < 0.4)
        sigma = [float(rng.uniform(0.05, 0.98) if flow else np.exp(rng.uniform(np.log(0.03), np.log(14.6)))) for _ in range(B)]
        if rng.random() < 0.5:
            sigma = [sigma[0]] * B
        cases.append(dict(id=k, shape=(B, Cc) + sp, flow=flow, sigma=sigma, n=int(rng.integers(0, 7)),
                          model=str(rng.choice(["identity", "two_heads", "bare", "one_tuple"])),
                          mask=str(rng.choice(["full", "chan", "batch1", "all0", "all1"])),
                          lam=float(rng.choice([0.1, 1.0, 5.0, 12.0])), beta=float(rng.choice([1.0, 0.5, 2.0])),
                          step=float(rng.choice([0.05, 0.2, 0.6])), min_frac=float(rng.choice([0.0, 0.3, 1.0])),
                          noncontig=bool(rng.random() < 0.2)))
    return cases


@pytest.mark.parametrize("c", _random_cases(48), ids=lambda c: f"r{c['id']}")
def test_randomized_configurations_match_oracle(c, cuda_device):
    from lanpaint_b200.engine import NoiseTape
    dev = cuda_device
    shape = c["shape"]
    g = torch.Generator().manual_seed(1000 + c["id"])
    x, y, noise = (torch.randn(shape, generator=g).to(dev) for _ in range(3))
    B, Cc = shape[0], shape[1]
    if c["mask"] == "all0":
        m = torch.zeros((B, 1) + shape[2:])
    elif c["mask"] == "all1":
        m = torch.ones((B, 1) + shape[2:])
    elif c["mask"] == "batch1":
        m = (torch.rand((1, 1) + shape[2:], generator=g) < 0.5).float()
    elif c["mask"] == "chan":
        m = (torch.rand((B, 1) + shape[2:], generator=g) < 0.5).float()
    else:
        m = (torch.rand(shape, generator=g) < 0.5).float()     # genuinely channel-dependent mask
    m = m.to(dev)
    mask_full = m.expand(shape).contiguous()
    sig = torch.tensor(c["sigma"], device=dev)
    times = O.times_from_sigma(sig, c["flow"])
    hp = O.Hyper(n_steps=c["n"], lam=c["lam"], beta=c["beta"], step_size=c["step"], min_step_frac=c["min_frac"],
                 flow=c["flow"])
    tape = O.NoiseTape(generator=torch.Generator().manual_seed(c["id"]))
    out_o, x_o = O.outer_step(make_model(c["model"], c["flow"]), x.clone(), y, noise, sig, mask_full, times, hp,
                              n_steps=c["n"], draw=tape)
    eng = _engine(make_model(c["model"], c["flow"]),
                  dict(n_steps=c["n"], lam=c["lam"], beta=c["beta"], step_size=c["step"], min_step_frac=c["min_frac"],
                       flow=c["flow"]), rng=NoiseTape(tape.recorded))
    xe = x.clone()
    if c["noncontig"] and xe.ndim >= 4:
        xe = xe.transpose(-1, -2).contiguous().transpose(-1, -2)
    out_e = eng(xe, y, noise, sig, m, tuple(times), {}, 0, n_steps=c["n"])
    tol = TIGHT * (10 if min(c["sigma"]) < 0.06 and not c["flow"] else 1)   # 1-abt ~ 1e-3: the reference's own
    assert max_rel(out_e, out_o) <= tol and max_rel(xe, x_o) <= tol, c       # cancellation noise grows there


def test_graph_statics_follow_the_tensor_not_the_address(cuda_device):
    """The caching allocator hands a freed tensor's address to the next one: operand caches must key on the
    tensor object, or a new request would silently reuse the previous request's clean latent."""
    from lanpaint_b200.runner import SynthDenoiser, VESampling
    dev = cuda_device
    shape = (2, 4, 32, 32)
    x, _, noise, m = synth_inputs(shape, seed=3, device=dev)
    sig = torch.full((2,), 2.0)
    times = tuple(O.times_from_sigma(sig, False))

    def run(eng, y):
        torch.manual_seed(1)
        return eng(x.clone(), y, noise, sig, m, times, None, 0, n_steps=3)

    eng = _engine(SynthDenoiser(VESampling()), dict(n_steps=3), rng="philox", cuda_graph=True, batched_replace="per_sample")
    y1 = torch.randn(shape, device=dev)
    out1 = run(eng, y1)
    ptr = y1.data_ptr()
    del y1
    y2 = torch.randn(shape, device=dev) + 3.0
    same_address = y2.data_ptr() == ptr
    out2 = run(eng, y2)
    want = run(_engine(SynthDenoiser(VESampling()), dict(n_steps=3), rng="philox", batched_replace="per_sample"), y2)
    assert torch.equal(out2, want) and not torch.equal(out1, out2), f"stale operand (same address: {same_address})"


def test_tma_staged_variant_is_bit_identical(cuda_device):
    """lp_set_option("tma", 1): the persistent cp.async.bulk/mbarrier variant of the steady kernel must produce
    exactly what the LDG variant does (same arithmetic, same Philox stream) -- including a ragged last tile."""
    from lanpaint_b200 import _native
    from lanpaint_b200.runner import SynthDenoiser, VESampling
    lib = _native.load()
    dev = cuda_device
    res = {}
    try:
        for shape in ((24, 4, 128, 128), (2, 16, 21, 80, 48)):      # S = 16384 (8 tiles) and S = 80640 (39.4 tiles)
            x, y, noise, m = synth_inputs(shape, seed=31, device=dev)
            sig = torch.full((shape[0],), 1.7)
            times = tuple(O.times_from_sigma(sig, False))
            for tma in (0, 1):
                assert lib.lp_set_option(b"tma", tma) == 0
                torch.manual_seed(17)
                eng = _engine(SynthDenoiser(VESampling()), dict(n_steps=4), rng="philox", batched_replace="per_sample")
                xx = x.clone()
                out = eng(xx, y, noise, sig, m, times, None, 0, n_steps=4)
                res[(shape, tma)] = (out, xx)
            assert torch.equal(res[(shape, 0)][0], res[(shape, 1)][0])
            assert torch.equal(res[(shape, 0)][1], res[(shape, 1)][1])
    finally:
        lib.lp_set_option(b"tma", 1)   # the default


def test_packed_box_muller_is_bit_identical_to_curands(cuda_device):
    """The torch-stream TMA kernel computes cuRAND's Box-Muller two at a time in FP32x2 (FFMA2) arithmetic with
    CUDA's logf / sqrtf specialised to the argument range.  Device self test: 2^28 pseudo-random input quadruples
    plus every combination of the extreme inputs, bitwise against the scalar cuRAND form."""
    from lanpaint_b200 import _native
    lib = _native.load()
    bad = torch.zeros(1, dtype=torch.int64, device=cuda_device)
    for seed in (1, 0xDEADBEEFCAFE):
        rc = lib.lp_selftest_box_muller(1 << 28, seed, C.c_void_p(bad.data_ptr()),
                                        C.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == 0
        assert int(bad.item()) == 0


def test_torch_stream_tma_variant_is_bit_identical(cuda_device):
    """The seed-exact stream at HBM-bound sizes runs substep_torch_tma_kernel (producer warp + cp.async.bulk slots,
    4 Philox subsequences per thread).  It must reproduce the LDG torch kernels bit for bit -- same randn stream,
    same arithmetic -- on SDXL batches, on a Wan-sized video latent whose channel size is not a multiple of the
    sub-tile (mask slices split at channel boundaries) and on a tensor that ends inside a plane."""
    from lanpaint_b200 import _native
    from lanpaint_b200.runner import SynthDenoiser, VESampling
    lib = _native.load()
    dev = cuda_device
    res = {}
    try:
        for shape in ((24, 4, 128, 128), (1, 16, 21, 80, 45), (5, 4, 128, 128), (8, 4, 96, 112)):
            x, y, noise, m = synth_inputs(shape, seed=33, device=dev)
            sig = torch.full((shape[0],), 1.3)
            times = tuple(O.times_from_sigma(sig, False))
            for tma in (0, 1):     # LDG kernels, TMA kernel
                assert lib.lp_set_option(b"tma", tma) == 0
                torch.manual_seed(23)
                eng = _engine(SynthDenoiser(VESampling()), dict(n_steps=4), rng="torch", batched_replace="per_sample")
                xx = x.clone()
                out = eng(xx, y, noise, sig, m, times, None, 0, n_steps=4)
                res[(shape, tma)] = (out, xx, torch.cuda.default_generators[dev.index or 0].get_offset())
            assert torch.equal(res[(shape, 0)][0], res[(shape, 1)][0]), shape
            assert torch.equal(res[(shape, 0)][1], res[(shape, 1)][1]), shape
            assert res[(shape, 0)][2] == res[(shape, 1)][2]
    finally:
        lib.lp_set_option(b"tma", 1)


@pytest.mark.parametrize("rng", ["philox", "torch"])
def test_tma_variants_with_fused_cfg_combine(rng, cuda_device):
    """cond / uncond fed straight to the TMA-staged kernels (>= 2^20 elements, lp_heads.combine) == the same run
    with the LDG kernels == the combines materialised by torch."""
    from lanpaint_b200 import _native
    from lanpaint_b200.engine import CfgPair
    from lanpaint_b200.runner import VESampling
    lib = _native.load()
    dev = cuda_device
    shape = (20, 4, 128, 128)     # 1.3 M elements
    x, y, noise, m = synth_inputs(shape, seed=35, device=dev)
    sig = torch.full((shape[0],), 2.1)
    times = tuple(O.times_from_sigma(sig, False))

    class Guider:
        def __init__(self, fused):
            self.inner_model = self
            self.model_sampling = VESampling()
            self.fused = fused

        def __call__(self, xx, t, model_options=None, seed=None):
            c, u = 0.7 * xx + 0.1 * torch.tanh(xx) + 0.3, 0.7 * xx + 0.1 * torch.tanh(xx) - 0.2
            pair = CfgPair(c, u, 4.5, -0.5)
            return pair if self.fused else pair.heads()
    res = {}
    try:
        for key, tma, fused in (("tma", 1, True), ("ldg", 0, True), ("eager", 1, False)):
            assert lib.lp_set_option(b"tma", tma) == 0
            torch.manual_seed(29)
            eng = _engine(Guider(fused), dict(n_steps=3), rng=rng, batched_replace="per_sample")
            xx = x.clone()
            out = eng(xx, y, noise, sig, m, times, None, 0, n_steps=3)
            res[key] = (out, xx)
        for k in ("ldg", "eager"):
            assert torch.equal(res["tma"][0], res[k][0]) and torch.equal(res["tma"][1], res[k][1]), k
    finally:
        lib.lp_set_option(b"tma", 1)


@pytest.mark.parametrize("combine,with_next,with_out", [(False, True, False), (False, True, True), (True, True, True),
                                                         (False, False, True), (True, False, False)])
def test_boundary_matches_torch(combine, with_next, with_out, cuda_device):
    """lp_boundary: the step boundary (epilogue + Euler update + next replace step, optional CFG combine) against
    plain torch, through the C ABI."""
    from lanpaint_b200 import _native
    from lanpaint_b200.schedule import Hyper, build_table
    lib = _native.load()
    dev = cuda_device
    B, Cc, S = 6, 4, 128 * 128 + 32 * 16
    shape = (B, Cc, S)
    gen = torch.Generator(device=dev).manual_seed(1)
    a, b, y, nz, x0 = (torch.randn(shape, device=dev, generator=gen) for _ in range(5))
    m8 = (torch.rand(B, 1, S, device=dev, generator=gen) < 0.5).to(torch.uint8)
    sig = torch.linspace(0.5, 3.0, B)
    ve, abt, _ = O.times_from_sigma(sig, False)
    tab = torch.from_numpy(build_table(abt.numpy(), ve.numpy(), Hyper(0.2, 5.0, 1.0, 1.0, False),
                                       rep_noise=sig.numpy(), rep_y=np.ones(B))).to(dev)
    dims = _native.Dims(B, Cc * S, S, S, 0, 0)
    P = C.c_void_p
    coef, cfg = -0.37, 3.5

    x1, o1 = x0.clone(), torch.full(shape, float("nan"), device=dev)
    h = _native.Heads(a.data_ptr(), b.data_ptr() if combine else None, _native.DTYPE_F32, 1 if combine else 0, cfg, cfg)
    rc = lib.lp_boundary(C.byref(h), P(y.data_ptr()), P(nz.data_ptr()) if with_next else None, P(m8.data_ptr()),
                         P(x1.data_ptr()), P(o1.data_ptr()) if with_out else None, C.c_float(coef),
                         P(tab.data_ptr()) if with_next else None, C.byref(dims),
                         P(torch.cuda.current_stream().cuda_stream))
    assert rc == 0
    known = m8.bool().expand(shape)
    d = b + (a - b) * cfg if combine else a
    o = torch.where(known, y, d)
    xe = torch.addcmul(x0, x0 - o, torch.tensor(coef, device=dev))
    if with_next:
        rn = tab[:, _native.T_INVS + 3].view(B, 1, 1)     # LP_T_REPN = 5
        ry = tab[:, _native.T_INVS + 4].view(B, 1, 1)
        xe = torch.where(known, rn * nz + ry * y, xe)
    assert (x1 - xe).abs().max().item() <= 1e-5 * max(1.0, xe.abs().max().item())
    if with_out:
        assert torch.equal(o1, o)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("rng_mode", ["tape", "philox", "torch"])
def test_half_precision_heads_are_read_in_kernel(dtype, rng_mode, cuda_device):
    """A model that returns bf16 / fp16 predictions: the kernels read them as they are and widen in registers
    (lp_heads.dtype) -- no .float() pass.  Reference semantics: type promotion to fp32 when x_t (fp32) meets the
    half-precision head (lanpaint.py:182-184), i.e. the oracle fed the same rounded heads."""
    from lanpaint_b200.engine import NoiseTape
    from lanpaint_b200.runner import SynthDenoiser, VESampling
    dev = cuda_device
    shape = (20, 4, 128, 128) if rng_mode != "tape" else (2, 4, 64, 64)
    x, y, noise, m = synth_inputs(shape, seed=41, device=dev)
    sig = torch.full((shape[0],), 1.9)
    times = tuple(O.times_from_sigma(sig, False))
    n = 3

    class Rounded:     # what the engine sees from a half-precision network, as an fp32-returning model
        def __init__(self, inner):
            self.inner, self.inner_model, self.model_sampling = inner, self, inner.model_sampling

        def __call__(self, xx, t, model_options=None, seed=None):
            return tuple(h.float() for h in self.inner(xx, t))
    if rng_mode == "tape":
        # Oracle and engine must see the SAME rounded heads, so the network here ignores its input and replays a
        # table of half-precision predictions (an input-dependent network would round differently wherever the two
        # implementations' fp32 model inputs differ in the last bit -- a 2^-8 jump in bf16).
        hp = O.Hyper(n_steps=n, min_step_frac=1.0)
        tape = O.NoiseTape(generator=torch.Generator().manual_seed(2))
        gh = torch.Generator().manual_seed(8)
        table = [(torch.randn(shape, generator=gh).to(dev).to(dtype), torch.randn(shape, generator=gh).to(dev).to(dtype))
                 for _ in range(n + 1)]

        class TableModel:
            def __init__(self):
                self.inner_model, self.model_sampling, self.calls = self, O.VESampling(), 0

            def __call__(self, xx, t, model_options=None, seed=None):
                self.calls += 1
                return table[self.calls - 1]
        want_out, want_x = O.outer_step(TableModel(), x.clone(), y, noise, sig.to(dev), m.expand(shape),
                                        O.times_from_sigma(sig.to(dev), False), hp, n_steps=n, draw=tape)
        eng = _engine(TableModel(), dict(n_steps=n), rng=NoiseTape([d.to(dev) for d in tape.recorded]))
        xx = x.clone()
        out = eng(xx, y, noise, sig, m, times, None, 0, n_steps=n)
        assert out.dtype == torch.float32 and max_rel(out, want_out) <= 2e-5 and max_rel(xx, want_x) <= 2e-5
        return
    res = {}
    for key in ("native", "widened"):
        torch.manual_seed(31)
        net = SynthDenoiser(VESampling(), dtype=dtype)
        eng = _engine(net if key == "native" else Rounded(net), dict(n_steps=n), rng=rng_mode, batched_replace="per_sample")
        xx = x.clone()
        res[key] = (eng(xx, y, noise, sig, m, times, None, 0, n_steps=n), xx)
    assert torch.equal(res["native"][0], res["widened"][0]) and torch.equal(res["native"][1], res["widened"][1])


def test_two_devices_in_one_process(cuda_device):
    """Per-device launch state (SM count, dynamic shared memory opt-in, torch's randn geometry) must follow the
    device of the tensors, not the first device the process touched (ComfyUI multi-GPU, thread-per-device replicas)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from lanpaint_b200.runner import SynthDenoiser, VESampling
    shape = (20, 4, 128, 128)     # large enough for the TMA-staged kernels (>48 KB dynamic shared memory)
    outs = {}
    for rng in ("philox", "torch"):
        for d in (0, 1):
            dev = torch.device("cuda", d)
            x, y, noise, m = synth_inputs(shape, seed=43, device=dev)
            sig = torch.full((shape[0],), 1.1)
            times = tuple(O.times_from_sigma(sig, False))
            torch.cuda.default_generators[d].manual_seed(5)
            eng = _engine(SynthDenoiser(VESampling()), dict(n_steps=3), rng=rng, batched_replace="per_sample")
            xx = x.clone()
            outs[(rng, d)] = (eng(xx, y, noise, sig, m, times, None, 0, n_steps=3).cpu(), xx.cpu())   # current device stays 0
        assert torch.equal(outs[(rng, 0)][0], outs[(rng, 1)][0]) and torch.equal(outs[(rng, 0)][1], outs[(rng, 1)][1])


# ----------------------------------------------------------------------------
# 9. size-independent property at BASELINE size: the fused update is affine in its operands
# ----------------------------------------------------------------------------
@pytest.mark.parametrize("flags", [1 | 2, 2, 0])      # first+fused next, steady, last
def test_update_is_affine_in_its_operands_at_full_size(flags, cuda_device):
    """For fixed mask and coefficients, one launch maps (x, x0, x0_BIG, y, C, xi1, xi2) affinely to (x', C'):
    f(u+v) - f(u) - f(v) + f(0) == 0.  Checked on [32,4,128,128] (BASELINE config 3) through the C ABI."""
    from lanpaint_b200 import _native
    from lanpaint_b200.schedule import Hyper, build_table
    lib = _native.load()
    dev = cuda_device
    B, Cc, S = 32, 4, 128 * 128
    shape = (B, Cc, S)
    sig = torch.linspace(0.05, 14.0, B)
    ve, abt, _ = O.times_from_sigma(sig, False)
    tab = torch.from_numpy(build_table(abt.numpy(), ve.numpy(), Hyper(0.2, 5.0, 1.0, 1.0, False))).to(dev)
    m8 = (torch.rand(B, 1, S, device=dev) < 0.5).to(torch.uint8)
    dims = _native.Dims(B, Cc * S, S, S, 0, 0)
    P = C.c_void_p
    gen = torch.Generator(device=dev).manual_seed(0)
    u = [torch.randn(shape, device=dev, generator=gen) for _ in range(7)]
    v = [torch.randn(shape, device=dev, generator=gen) for _ in range(7)]

    def f(ops):
        x, x0, x0b, y, c, t0, t1 = (t.clone() for t in ops)
        r = _native.Rng(mode=_native.RNG_TAPE, tape0=t0.data_ptr(), tape1=t1.data_ptr())
        rc = lib.lp_substep_f32(P(x.data_ptr()), P(x0.data_ptr()), P(x0b.data_ptr()), P(y.data_ptr()), P(m8.data_ptr()),
                                P(c.data_ptr()), None, None, P(tab.data_ptr()), C.byref(dims), C.byref(r),
                                flags | 4, P(torch.cuda.current_stream().cuda_stream))
        assert rc == 0
        return x.double(), c.double()

    zero = [torch.zeros(shape, device=dev) for _ in range(7)]
    fu, fv, fuv, f0 = f(u), f(v), f([a + b for a, b in zip(u, v)]), f(zero)
    for k in range(2):
        resid = (fuv[k] - fu[k] - fv[k] + f0[k]).abs().max().item()
        scale = max(fuv[k].abs().max().item(), 1.0)
        assert resid <= 2e-5 * scale, (k, resid, scale)
    assert f0[0].abs().max().item() == 0.0 and f0[1].abs().max().item() == 0.0   # and linear: f(0) = 0
