"""oracle/_ref (the reference's own engine, compiled to bytecode by oracle/build_ref.py) against the oracle port:
the thing bench.py times as `cpu_baseline.kind == "reference"` is the code the port restates, bit for bit.  The
reference engine's outputs for the same cases are also stored (tests/golden/aux_ref_port_cases.npz, written by
tests/golden/make_golden.py --ref-port), so the port is held to them where oracle/_ref is not built."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN_DIR
from oracle import build_ref
from oracle import langevin_oracle as O

CASES = [(False, 5, 1), (False, 3, 2), (True, 4, 1)]


def port_case(flow, n, batch):
    """-> (engine arguments, the port's (out, x), its noise tape) of one case."""
    g = torch.Generator().manual_seed(3)
    shape = (batch, 4, 16, 16)
    x, y, noise = (torch.randn(shape, generator=g) for _ in range(3))
    mask = (torch.rand((batch, 1, 16, 16), generator=g) < 0.5).float().expand(shape).contiguous()
    sigma = torch.full((batch,), 0.6 if flow else 2.5)
    times = O.times_from_sigma(sigma, flow)
    hp = O.Hyper(n_steps=n, min_step_frac=1.0, flow=flow)
    tape = O.NoiseTape(generator=torch.Generator().manual_seed(4))
    sampling = O.FlowSampling() if flow else O.VESampling()
    want = O.outer_step(O.PointwiseDenoiser(sampling), x.clone(), y, noise, sigma, mask, times, hp, n_steps=n, draw=tape)
    return (x, y, noise, sigma, mask, times, hp), want, tape.recorded


def run_reference(Ref, flow, n, args, draws, monkeypatch):
    """The reference engine class `Ref` on one case, its torch.randn_like replaying `draws` -> (out, x)."""
    x, y, noise, sigma, mask, times, hp = args
    replay = iter(draws)
    monkeypatch.setattr(torch, "randn_like", lambda t, **kw: next(replay).to(t.dtype))
    sampling = O.FlowSampling() if flow else O.VESampling()
    eng = Ref(O.PointwiseDenoiser(sampling), n, 15.0, hp.lam, hp.beta, hp.step_size, IS_FLUX=False, IS_FLOW=flow,
              MinStepFrac=1.0)
    xr = x.clone()
    out = eng(xr, y, noise, sigma, mask, tuple(times), {}, 0, n_steps=n)
    return out, xr


@pytest.mark.parametrize("flow,n,batch", CASES)
def test_reference_bytecode_equals_the_port(flow, n, batch, monkeypatch):
    args, (want_out, want_x), draws = port_case(flow, n, batch)
    z = np.load(os.path.join(GOLDEN_DIR, "aux_ref_port_cases.npz"))
    key = f"{int(flow)}_{n}_{batch}"
    assert torch.equal(torch.from_numpy(z[key + "_out"]), want_out) and torch.equal(torch.from_numpy(z[key + "_x"]), want_x)
    Ref = build_ref.load()
    if Ref is None:
        return          # the stored outputs above are the reference's; the live comparison needs oracle/_ref
    out, xr = run_reference(Ref, flow, n, args, draws, monkeypatch)
    assert torch.equal(out, want_out) and torch.equal(xr, want_x)


def test_reference_bytecode_node_layer_reproduces_the_node_goldens(monkeypatch):
    """oracle/_ref's node layer (what `bench.py --impl reference` calls) is the code that wrote tests/golden/node_*.npz:
    the same call on this host reproduces a fixture (to fp32 round-off: the host's tanh may differ by an ulp from the
    build container's)."""
    import contextlib
    import io
    import json
    import os
    import sys

    import numpy as np

    from _node_cases import build_patcher, call_node
    from conftest import GOLDEN_DIR
    ref_nodes = build_ref.load_nodes()
    if ref_nodes is None:
        pytest.skip("oracle/_ref not built (needs /root/reference: `make -C oracle`)")
    assert ref_nodes.__file__.endswith(".pyc")
    for name in ("node_ksampler_prompt_first_batch2", "node_advanced_window_leftover", "node_custom_random_noise"):
        z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
        c = json.loads(str(z["meta"]))
        replay = iter(torch.from_numpy(t.astype(np.float32)) for t in z["tape"])
        monkeypatch.setattr(torch, "randn_like", lambda t, **kw: next(replay).to(t.dtype))
        if "noise_image" in z.files:
            image = torch.from_numpy(z["noise_image"])
            monkeypatch.setattr(sys.modules["comfy.sample"], "prepare_noise", lambda *a, **k: image.clone())
        latent = {"samples": torch.from_numpy(z["samples"]),
                  "noise_mask": torch.from_numpy(z["noise_mask"].astype(np.float32))}
        with contextlib.redirect_stdout(io.StringIO()):
            outs = call_node(ref_nodes, c, build_patcher(c), latent)
        want = torch.from_numpy(z["out"])
        assert float((outs[0]["samples"] - want).abs().max() / want.abs().max()) <= 1e-6
        assert next(replay, None) is None, "the reference consumed fewer draws than the fixture holds"
