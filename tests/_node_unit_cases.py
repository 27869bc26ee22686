"""Unit-level calls into a node module, shared by tests/golden/make_golden.py --node-units (which makes them on the
REFERENCE's nodes.py and stores the answers in tests/golden/node_unit_answers.json) and
tests/test_reference_suite_on_b200_nodes.py (which makes them on lanpaint_b200/comfy_nodes.py and compares).

The calls are the ones the reference's own node-layer tests make (tests/test_node_params.py, test_min_step_frac.py,
test_reshape_mask.py and the detection / guarded-import part of test_av_schedule.py): the widget surface and the
retired hidden inputs, the value sanitiser, the MinStepFrac inner-step ramp, reshape_mask / prepare_mask incl. the
video temporal union, MiniMax-H3 AV-pack detection.  The module is imported under the bare ComfyUI stubs those tests
install (no ComfyUI, no minicomfy), so importing it there is part of what is checked.  Test infrastructure."""
import sys
import types

import torch

CLASSES = ("LanPaint_KSampler", "LanPaint_KSamplerAdvanced", "LanPaint_SamplerCustom", "LanPaint_SamplerCustomAdvanced")


def install_comfy_stubs(version="0.6.0"):
    """The module surface a node module imports, as ComfyUI-less tooling stubs it (replaces what is in sys.modules)."""
    def stub(name, **attrs):
        m = types.ModuleType(name)
        for k, v in attrs.items():
            setattr(m, k, v)
        sys.modules[name] = m
        return m

    def repeat_to_batch_size(t, n):  # comfy.utils.repeat_to_batch_size semantics
        if t.shape[0] >= n:
            return t[:n]
        reps = (n + t.shape[0] - 1) // t.shape[0]
        return t.repeat((reps,) + (1,) * (t.ndim - 1))[:n]

    comfy = stub("comfy")
    comfy.__path__ = []
    comfy.utils = stub("comfy.utils", repeat_to_batch_size=repeat_to_batch_size)
    comfy.samplers = stub("comfy.samplers", KSAMPLER=type("KSAMPLER", (), {}),
                          KSampler=type("KSampler", (), {"SCHEDULERS": ["<SCHEDULERS>"]}))
    comfy.model_base = stub("comfy.model_base", ModelType=types.SimpleNamespace(FLUX="FLUX", FLOW="FLOW"),
                            WAN22=type("WAN22", (), {}))
    stub("nodes")
    stub("latent_preview")
    stub("comfyui_version", __version__=version)


def _tensor(t):
    return {"shape": list(t.shape), "device": t.device.type, "values": t.contiguous().flatten().tolist()}


def _plain(v):
    """JSON-able form that keeps the type apart (True vs 1, 5 vs 5.0, tuple layouts as lists)."""
    if isinstance(v, (list, tuple)):
        return [_plain(x) for x in v]
    return {"type": type(v).__name__, "value": v}


class _Diffusion:
    sigma_shift_video = 12.0
    sigma_shift_audio = 3.0


def _patcher(with_shifts):
    model = types.SimpleNamespace(diffusion_model=_Diffusion()) if with_shifts else object()
    return types.SimpleNamespace(model=model)


def run(nodes):
    """-> JSON-able answers of node module `nodes` to every call."""
    out = {"widgets": {}}
    for name in CLASSES:
        spec = getattr(nodes, name).INPUT_TYPES()
        out["widgets"][name] = {"required": list(spec.get("required", {})), "hidden": list(spec.get("hidden", {}))}

    modes = ("Image First", "Prompt First")
    sanitize = [("Image First", "Image First", modes), ("Prompt First", "Image First", modes), (1.0, "Image First", modes),
                ("bogus", "Image First", modes), (None, "Image First", modes),
                (5, 5, None), (3.7, 0.2, None), ("abc", 0.2, None), (None, 0.2, None), (True, 5, None), (7, 0.2, None)]
    out["sanitize"] = [_plain(nodes._sanitize_param(v, d, allowed=a)) for v, d, a in sanitize]

    ramp = [(n, f, m) for n in (0, 1, 5, 10) for m in (0.0, 0.05, 0.2)
            for f in (0.0, 0.005, 0.01, 0.025, 0.04, 0.05, 0.1, 0.2, 0.5)]
    out["min_step_frac"] = [[n, f, m, _plain(nodes.min_step_frac_effective_steps(n, f, m))] for n, f, m in ramp]

    strokes = torch.zeros(8, 8, 8)
    strokes[2, 5, 5] = 1.0
    strokes[6, 7, 7] = 1.0
    unpicked = torch.zeros(8, 8, 8)
    unpicked[3, 5, 5] = 1.0
    short = torch.zeros(3, 8, 8)
    short[1, 5, 5] = 1.0
    reshape = {"bhw_to_5d": (torch.zeros(1, 4, 4), (1, 16, 1, 8, 8), False),
               "video_picked_frames": (strokes, (1, 16, 2, 4, 4), True),
               "video_unpicked_frame": (unpicked, (1, 16, 2, 4, 4), True),
               "video_short_sequence": (short, (1, 16, 1, 4, 4), True)}
    out["reshape_mask"] = {k: _tensor(nodes.reshape_mask(m, s, video_inpainting=v)) for k, (m, s, v) in reshape.items()}
    out["prepare_mask_hw"] = _tensor(nodes.prepare_mask(torch.zeros(4, 4), (2, 3, 8, 8), device=torch.device("cpu"),
                                                        video_inpainting=False))

    two = [(1, 24, 37, 30, 54), (1, 32, 2, 207)]
    over = {"transformer_options": {"minimax_h3_sigma_shift_video": 10.0, "minimax_h3_sigma_shift_audio": 2.5}}
    detect = {"single_stream": (True, {}, [two[0]]), "no_shapes": (True, {}, None), "no_shift_attrs": (False, {}, two),
              "av_pack": (True, {}, two), "node_overrides": (True, over, two)}
    out["detect_minimax_h3"] = {k: _plain(nodes._detect_minimax_h3_audio(_patcher(s), o, shapes))
                                for k, (s, o, shapes) in detect.items()}
    out["time_shift_sigma_is_none"] = nodes.time_shift_sigma is None
    return out
