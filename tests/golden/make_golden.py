"""Generate golden vectors from the REAL reference engine (run in the build container only).

    python tests/golden/make_golden.py            # writes every fixture under tests/golden/
    python tests/golden/make_golden.py --engine   # or one family: --engine | --api | --node-units | --ref-port | --earlystop | --av

The reference (`/root/reference/src/LanPaint/lanpaint.py`, imported unmodified)
is driven with stand-in denoisers that follow its own test doubles' protocol
(tests/test_av_schedule.py:110-130) and with `torch.randn_like` patched to a
recorded noise tape, so every fixture carries: the inputs, the tape, the
returned `out`, and the in-place-rewritten `x`.  `/root/reference` does not
exist on the GPU box, so nothing but this script reads it.

Node-level fixtures (the reference's own nodes.py driven over minicomfy: node_*.npz) come from the sibling script
tests/golden/make_node_golden.py.

Fixture format (npz): x, y, noise, sigma, mask, ve, abt, flow_t, tape[k,...],
out, x_new, meta (json string: hyper-parameters, model kind, n_steps, flags).
"""
from __future__ import annotations

import json
import os
import sys
import zlib
from unittest import mock

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, "/root/reference")

from oracle import langevin_oracle as O  # noqa: E402
from src.LanPaint.lanpaint import LanPaint as RefEngine  # noqa: E402


def make_model(kind: str, flow: bool):
    sampling = O.FlowSampling() if flow else O.VESampling()
    if kind == "identity":
        return O.IdentityDenoiser(sampling)
    if kind == "two_heads":
        return O.PointwiseDenoiser(sampling)
    if kind == "bare":
        return O.PointwiseDenoiser(sampling, heads=0)
    if kind == "one_tuple":
        return O.PointwiseDenoiser(sampling, heads=1)
    raise KeyError(kind)


CASES = [
    # name, shape, flow, model, n_steps, sigma, density(known fraction), lam, beta, step, min_frac, zero_noise
    dict(name="cfg1_ve_identity_n5", shape=(1, 4, 64, 64), flow=False, model="identity", n=5, sigma=[2.0], dens=0.5),
    dict(name="ve_two_heads_n5", shape=(1, 4, 16, 16), flow=False, model="two_heads", n=5, sigma=[2.0], dens=0.5),
    dict(name="ve_two_heads_n1", shape=(1, 4, 16, 16), flow=False, model="two_heads", n=1, sigma=[7.5], dens=0.5),
    dict(name="ve_two_heads_n2", shape=(1, 4, 16, 16), flow=False, model="two_heads", n=2, sigma=[0.3], dens=0.3),
    dict(name="ve_two_heads_n0", shape=(1, 4, 16, 16), flow=False, model="two_heads", n=0, sigma=[1.0], dens=0.5),
    dict(name="ve_two_heads_n10_lowsigma", shape=(1, 4, 16, 16), flow=False, model="two_heads", n=10, sigma=[0.05], dens=0.5),
    dict(name="ve_bare_n3", shape=(1, 4, 16, 16), flow=False, model="bare", n=3, sigma=[14.6146], dens=0.5),
    dict(name="ve_one_tuple_n3", shape=(1, 4, 16, 16), flow=False, model="one_tuple", n=3, sigma=[1.3], dens=0.9),
    dict(name="ve_mask_all_known", shape=(1, 4, 16, 16), flow=False, model="two_heads", n=3, sigma=[2.0], dens=1.0),
    dict(name="ve_mask_none_known", shape=(1, 4, 16, 16), flow=False, model="two_heads", n=3, sigma=[2.0], dens=0.0),
    dict(name="ve_engine_default_minfrac0", shape=(1, 4, 16, 16), flow=False, model="two_heads", n=4, sigma=[0.8], dens=0.5, min_frac=0.0),
    dict(name="ve_hyper_variants", shape=(1, 4, 16, 16), flow=False, model="two_heads", n=4, sigma=[3.0], dens=0.5, lam=8.0, beta=1.5, step=0.15, min_frac=0.4),
    dict(name="ve_zero_noise_regen", shape=(1, 4, 16, 16), flow=False, model="two_heads", n=2, sigma=[2.0], dens=0.5, zero_noise=True),
    dict(name="ve_batch2_flowform_replace", shape=(2, 4, 16, 16), flow=False, model="two_heads", n=3, sigma=[2.0, 2.0], dens=0.5),
    dict(name="ve_batch3_mixed_sigma", shape=(3, 4, 8, 8), flow=False, model="two_heads", n=3, sigma=[0.4, 2.0, 9.0], dens=0.5),
    dict(name="flow_two_heads_n5", shape=(1, 16, 8, 8), flow=True, model="two_heads", n=5, sigma=[0.6], dens=0.5),
    dict(name="flow_identity_n3_high_t", shape=(1, 16, 8, 8), flow=True, model="identity", n=3, sigma=[0.97], dens=0.5),
    dict(name="flow_batch2", shape=(2, 16, 8, 8), flow=True, model="two_heads", n=3, sigma=[0.5, 0.5], dens=0.2),
    dict(name="video5d_flow_n3", shape=(1, 16, 3, 6, 5), flow=True, model="two_heads", n=3, sigma=[0.7], dens=0.5),
    dict(name="odd_size_ve_n3", shape=(1, 3, 5, 7), flow=False, model="two_heads", n=3, sigma=[1.1], dens=0.5),
]


def run_case(c: dict, seed: int = 0):
    g = torch.Generator().manual_seed(seed + zlib.crc32(c["name"].encode()) % 1000)  # stable across processes
    shape = tuple(c["shape"])
    flow = c["flow"]
    x = torch.randn(shape, generator=g)
    y = torch.randn(shape, generator=g)
    noise = torch.zeros(shape) if c.get("zero_noise") else torch.randn(shape, generator=g)
    mshape = (shape[0], 1) + shape[2:]
    dens = c["dens"]
    if dens >= 1.0:
        mask = torch.ones(mshape)
    elif dens <= 0.0:
        mask = torch.zeros(mshape)
    else:
        mask = (torch.rand(mshape, generator=g) < dens).float()
    mask = mask.expand(shape).contiguous()
    sigma = torch.tensor(c["sigma"], dtype=torch.float32)
    times = O.times_from_sigma(sigma, flow)
    hp = O.Hyper(n_steps=c["n"], lam=c.get("lam", 5.0), beta=c.get("beta", 1.0),
                 step_size=c.get("step", 0.2), min_step_frac=c.get("min_frac", 1.0), flow=flow)

    # ---- the real reference, noise drawn through a recording tape ----
    tape = O.NoiseTape(generator=torch.Generator().manual_seed(1234 + seed))
    model = make_model(c["model"], flow)
    eng = RefEngine(model, NSteps=hp.n_steps, Friction=hp.friction, Lambda=hp.lam, Beta=hp.beta,
                    StepSize=hp.step_size, IS_FLUX=False, IS_FLOW=flow, MinStepFrac=hp.min_step_frac)
    x_ref = x.clone()
    with mock.patch.object(torch, "randn_like", tape):
        out_ref = eng(x_ref, y, noise, sigma, mask, tuple(times), model_options={}, seed=0, n_steps=c["n"])
    draws = tape.recorded

    # ---- the oracle on the same tape must agree bit for bit ----
    replay = O.NoiseTape(draws)
    out_o, x_o = O.outer_step(make_model(c["model"], flow), x.clone(), y, noise, sigma, mask, times, hp,
                              n_steps=c["n"], draw=replay)
    assert replay.pos == len(draws), (replay.pos, len(draws))
    exact = torch.equal(out_o, out_ref) and torch.equal(x_o, x_ref)
    err = max(float((out_o - out_ref).abs().max()), float((x_o - x_ref).abs().max()))
    print(f"{c['name']:36s} draws={len(draws):2d} oracle==reference: {exact} (max abs diff {err:.2e})")
    assert err < 1e-6, c["name"]

    meta = dict(name=c["name"], flow=flow, model=c["model"], n_steps=c["n"], lam=hp.lam, beta=hp.beta,
                step_size=hp.step_size, min_step_frac=hp.min_step_frac, friction=hp.friction,
                n_draws=len(draws), oracle_bit_exact=bool(exact), generator="reference@/root/reference lanpaint.py")
    tape_arr = np.stack([d.numpy() for d in draws]) if draws else np.zeros((0,) + shape, np.float32)
    np.savez_compressed(
        os.path.join(HERE, c["name"] + ".npz"),
        x=x.numpy(), y=y.numpy(), noise=noise.numpy(), sigma=sigma.numpy(),
        mask=mask[:, :1].numpy().astype(np.uint8), ve=times.ve_sigma.numpy(), abt=times.abt.numpy(),
        flow_t=times.flow_t.numpy(), tape=tape_arr, out=out_ref.numpy(), x_new=x_ref.numpy(),
        meta=np.array(json.dumps(meta)))


def main():
    torch.set_num_threads(1)
    for c in CASES:
        run_case(c)


# --------------------------------------------------------------------------------------------
# node API dump: INPUT_TYPES / RETURN_TYPES / ... of the reference's four sampler nodes
# --------------------------------------------------------------------------------------------
RESHAPE_CASES = {
    "img2d": ((64, 48), (2, 4, 8, 6), False),
    "img3d": ((1, 64, 64), (1, 16, 8, 8), False),
    "img4d": ((1, 1, 40, 40), (1, 4, 10, 10), False),
    "img_to_5d": ((64, 64), (1, 16, 3, 8, 8), False),
    "vid_frames_on_batch": ((17, 1, 32, 32), (1, 16, 5, 4, 4), True),
    "vid_raw_fhw": ((17, 32, 32), (1, 16, 5, 4, 4), True),
    "vid_still": ((32, 32), (1, 16, 5, 4, 4), True),
}


def dump_node_api():
    import importlib
    from _node_unit_cases import install_comfy_stubs
    install_comfy_stubs()
    ref = importlib.import_module("src.LanPaint.nodes")
    api = {}
    for name in ("LanPaint_KSampler", "LanPaint_KSamplerAdvanced", "LanPaint_SamplerCustom",
                 "LanPaint_SamplerCustomAdvanced"):
        cls = ref.NODE_CLASS_MAPPINGS[name]
        api[name] = {
            "INPUT_TYPES": cls.INPUT_TYPES(),
            "RETURN_TYPES": list(cls.RETURN_TYPES),
            "RETURN_NAMES": list(getattr(cls, "RETURN_NAMES", ())),
            "FUNCTION": cls.FUNCTION,
            "CATEGORY": cls.CATEGORY,
            "display_name": ref.NODE_DISPLAY_NAME_MAPPINGS[name],
        }
    api["KSAMPLER_NAMES"] = list(ref.KSAMPLER_NAMES)
    # reshape_mask known answers (mask prep runs once per sample; kept for drop-in behaviour)
    g = torch.Generator().manual_seed(7)
    cases = {}
    for key, (mshape, oshape, video) in RESHAPE_CASES.items():
        m = (torch.rand(mshape, generator=g) > 0.6).float()
        cases["in_" + key] = m.numpy()
        cases["out_" + key] = ref.reshape_mask(m, oshape, video).contiguous().numpy()
    np.savez_compressed(os.path.join(HERE, "aux_reshape_mask_cases.npz"), **cases)
    with open(os.path.join(HERE, "node_api.json"), "w") as f:
        json.dump(api, f, indent=1, ensure_ascii=False, sort_keys=False)
    for n in ("comfy", "comfy.utils", "comfy.samplers", "comfy.model_base", "nodes", "latent_preview",
              "comfyui_version", "src.LanPaint.nodes"):
        sys.modules.pop(n, None)
    print("node_api.json written")


def dump_ref_port():
    """The reference engine's outputs on tests/test_oracle_ref.py's cases (same inputs, same noise tape)."""
    import pytest
    import test_oracle_ref as T
    arrays = {}
    for flow, n, batch in T.CASES:
        args, _, draws = T.port_case(flow, n, batch)
        with pytest.MonkeyPatch.context() as mp:
            out, x = T.run_reference(RefEngine, flow, n, args, draws, mp)
        arrays[f"{int(flow)}_{n}_{batch}_out"], arrays[f"{int(flow)}_{n}_{batch}_x"] = out.numpy(), x.numpy()
    np.savez_compressed(os.path.join(HERE, "aux_ref_port_cases.npz"), **arrays)
    print("aux_ref_port_cases.npz written")


def dump_node_units():
    """The reference node module's answers to the unit-level calls of tests/_node_unit_cases.py."""
    import importlib
    import _node_unit_cases
    _node_unit_cases.install_comfy_stubs()
    ref = importlib.import_module("src.LanPaint.nodes")
    with open(os.path.join(HERE, "node_unit_answers.json"), "w") as f:
        json.dump(_node_unit_cases.run(ref), f, separators=(",", ":"))
        f.write("\n")
    for n in ("comfy", "comfy.utils", "comfy.samplers", "comfy.model_base", "nodes", "latent_preview",
              "comfyui_version", "src.LanPaint.nodes"):
        sys.modules.pop(n, None)
    print("node_unit_answers.json written")




# --------------------------------------------------------------------------------------------
# early-stop goldens: the reference's LanPaintEarlyStopper driven through LanPaint.__call__
# --------------------------------------------------------------------------------------------
def _custom_distance(prev, cur, ctx):
    return ((cur - prev) ** 2).mean()


EARLYSTOP_CASES = [
    dict(name="aux_es_midway", sigma=0.3, stop={"threshold": 0.3, "patience": 2}, n=10),
    dict(name="aux_es_immediate", sigma=1.0, stop={"threshold": 1e3, "patience": 1}, n=10),
    dict(name="aux_es_never", sigma=2.0, stop={"threshold": 1e-9, "patience": 1}, n=6),
    dict(name="aux_es_min_steps_legacy", sigma=1.0, stop={"threshold": 1e3, "patience": 1, "min_steps": 4}, n=10),
    dict(name="aux_es_custom_fn", sigma=1.0, stop={"threshold": 0.5, "patience": 1, "distance_fn": "mean_sq_xt"}, n=10),
    dict(name="aux_es_ctor_threshold", sigma=0.3, stop=None, ctor_threshold=0.26, ctor_patience=1, n=10),
]


def dump_earlystop():
    torch.set_num_threads(1)
    for c in EARLYSTOP_CASES:
        g = torch.Generator().manual_seed(11)
        shape = (1, 4, 16, 16)
        x = torch.randn(shape, generator=g)
        y = torch.randn(shape, generator=g)
        noise = torch.randn(shape, generator=g)
        mask = (torch.rand((1, 1, 16, 16), generator=g) < 0.5).float().expand(shape).contiguous()
        sigma = torch.tensor([c["sigma"]])
        times = O.times_from_sigma(sigma, False)
        tape = O.NoiseTape(generator=torch.Generator().manual_seed(2))
        model = make_model("two_heads", False)
        eng = RefEngine(model, NSteps=c["n"], Friction=15.0, Lambda=5.0, Beta=1.0, StepSize=0.2, MinStepFrac=1.0,
                        EarlyStopThreshold=c.get("ctor_threshold", 0.0), EarlyStopPatience=c.get("ctor_patience", 1))
        trace = []
        mo = {"lanpaint_semantic_trace": trace, "bench_case_id": c["name"], "bench_outer_step": 3, "bench_timestep": 0.5}
        if c["stop"] is not None:
            stop = dict(c["stop"])
            if stop.get("distance_fn") == "mean_sq_xt":
                stop["distance_fn"] = _custom_distance
            mo["lanpaint_semantic_stop"] = stop
        x_ref = x.clone()
        with mock.patch.object(torch, "randn_like", tape):
            out = eng(x_ref, y, noise, sigma, mask, tuple(times), model_options=mo, seed=0, n_steps=c["n"])
        meta = dict(name=c["name"], n_steps=c["n"], stop=c["stop"], ctor_threshold=c.get("ctor_threshold", 0.0),
                    ctor_patience=c.get("ctor_patience", 1), trace=trace, model_calls=model.calls,
                    n_draws=len(tape.recorded))
        print(f"{c['name']:28s} sub-steps run {len(trace):2d}/{c['n']} model calls {model.calls:2d} "
              f"dists {[round(t['dist'], 4) for t in trace][:6]}")
        np.savez_compressed(os.path.join(HERE, c["name"] + ".npz"), x=x.numpy(), y=y.numpy(), noise=noise.numpy(),
                            sigma=sigma.numpy(), mask=mask[:, :1].numpy().astype(np.uint8), ve=times.ve_sigma.numpy(),
                            abt=times.abt.numpy(), flow_t=times.flow_t.numpy(),
                            tape=np.stack([d.numpy() for d in tape.recorded]), out=out.numpy(), x_new=x_ref.numpy(),
                            meta=np.array(json.dumps(meta)))




# --------------------------------------------------------------------------------------------
# MiniMax-H3 AV per-row schedule goldens (lanpaint.py:60-74,173-180): flat pack [1,C,N], the last
# N - video_n positions are audio rows with their own (VE, abt, flow t) and target correction c
# --------------------------------------------------------------------------------------------
AV_CASES = [
    dict(name="aux_av_flat_n3", shape=(1, 1, 64), video_n=40, n=3, sigma=0.6, sigma_a=0.35, corr=0.625),
    dict(name="aux_av_flat_n0", shape=(1, 1, 64), video_n=40, n=0, sigma=0.5, sigma_a=0.2, corr=None),
    dict(name="aux_av_channels_n4", shape=(1, 4, 48), video_n=32, n=4, sigma=0.8, sigma_a=0.55, corr=0.8),
    dict(name="aux_av_odd_split_n2", shape=(1, 1, 37), video_n=21, n=2, sigma=0.4, sigma_a=0.3, corr=1.3),
]


def dump_av():
    torch.set_num_threads(1)
    for c in AV_CASES:
        g = torch.Generator().manual_seed(5)
        shape = c["shape"]
        x, y, noise = (torch.randn(shape, generator=g) for _ in range(3))
        mask = (torch.rand(shape, generator=g) < 0.5).float()
        sigma = torch.tensor([c["sigma"]])
        times = O.times_from_sigma(sigma, True)
        sig_a = torch.tensor([c["sigma_a"]])
        times_a = O.times_from_sigma(sig_a, True)
        ai = torch.zeros((1, 1, shape[-1]))
        ai[..., c["video_n"]:] = 1.0
        corr = None if c["corr"] is None else (1.0 - ai) + c["corr"] * ai
        tape = O.NoiseTape(generator=torch.Generator().manual_seed(3))
        model = make_model("two_heads", True)
        eng = RefEngine(model, NSteps=c["n"], Friction=15.0, Lambda=5.0, Beta=1.0, StepSize=0.2, IS_FLOW=True,
                        MinStepFrac=1.0)
        x_ref = x.clone()
        with mock.patch.object(torch, "randn_like", tape):
            out = eng(x_ref, y, noise, sigma, mask, tuple(times), model_options={}, seed=0, n_steps=c["n"],
                      current_times_audio=tuple(times_a), audio_indicator=ai, audio_correction=corr)
        # the oracle's AV path must agree with the reference bit for bit as well
        replay = O.NoiseTape(tape.recorded)
        hp = O.Hyper(n_steps=c["n"], min_step_frac=1.0, flow=True)
        out_o, x_o = O.outer_step(make_model("two_heads", True), x.clone(), y, noise, sigma, mask, times, hp,
                                  n_steps=c["n"], draw=replay, audio=O.Audio(ai, times_a, corr))
        exact = torch.equal(out_o, out) and torch.equal(x_o, x_ref)
        print(f"{c['name']:24s} draws {len(tape.recorded)} oracle==reference {exact}")
        assert exact
        meta = dict(name=c["name"], n_steps=c["n"], video_n=c["video_n"], corr=c["corr"], n_draws=len(tape.recorded))
        np.savez_compressed(os.path.join(HERE, c["name"] + ".npz"), x=x.numpy(), y=y.numpy(), noise=noise.numpy(),
                            sigma=sigma.numpy(), mask=mask.numpy().astype(np.uint8), ve=times.ve_sigma.numpy(),
                            abt=times.abt.numpy(), flow_t=times.flow_t.numpy(), ve_a=times_a.ve_sigma.numpy(),
                            abt_a=times_a.abt.numpy(), flow_a=times_a.flow_t.numpy(),
                            tape=np.stack([d.numpy() for d in tape.recorded]) if tape.recorded else np.zeros((0,) + shape, np.float32),
                            out=out.numpy(), x_new=x_ref.numpy(), meta=np.array(json.dumps(meta)))


if __name__ == "__main__":
    # python tests/golden/make_golden.py            -> everything
    # python tests/golden/make_golden.py --engine   -> only the engine cases (likewise --api, --node-units, --ref-port,
    #                                                   --earlystop, --av)
    picked = [a for a in sys.argv[1:] if a.startswith("--")]
    todo = {"--engine": main, "--api": dump_node_api, "--node-units": dump_node_units, "--ref-port": dump_ref_port,
            "--earlystop": dump_earlystop, "--av": dump_av}
    for flag, fn in todo.items():
        if not picked or flag in picked:
            fn()
