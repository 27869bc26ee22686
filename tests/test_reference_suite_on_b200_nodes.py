"""The REFERENCE's own unit-level node tests, restated as calls on `lanpaint_b200/comfy_nodes.py` and compared with
the answers the reference's node module gives to the same calls (tests/golden/node_unit_answers.json, written by
tests/golden/make_golden.py --node-units; the calls are in tests/_node_unit_cases.py).  They cover b1 of SURVEY 8b the
way the reference's CI does: the widget surface and the retired hidden inputs (its tests/test_node_params.py), the
value sanitiser, the MinStepFrac inner-step ramp (tests/test_min_step_frac.py), reshape_mask / prepare_mask incl. the
video temporal union (tests/test_reshape_mask.py), MiniMax-H3 AV-pack detection and the guarded optional imports
(tests/test_av_schedule.py; its numeric tests drive the reference ENGINE's internals and are covered by the engine
goldens).  Also here: the package imports and lists its nodes with no ComfyUI at all, as node-diff CI needs (reference
tests/test_LanPaint.py, __init__.py:14-98)."""
import json
import os
import subprocess
import sys

from conftest import GOLDEN_DIR, ROOT


def test_reference_node_tests_pass_on_this_node_module(tmp_path):
    """In a clean interpreter with only the bare ComfyUI stubs the reference's tests install (no ComfyUI, no
    minicomfy), import the node module and make every call; the answers must equal the reference's."""
    code = (
        "import importlib, json, sys\n"
        f"sys.path[:0] = [{ROOT!r}, {os.path.join(ROOT, 'tests')!r}]\n"
        "import _node_unit_cases as C\n"
        "C.install_comfy_stubs()\n"
        "nodes = importlib.import_module('lanpaint_b200.comfy_nodes')\n"
        "print(json.dumps({'file': nodes.__file__, 'answers': C.run(nodes)}))\n")
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=str(tmp_path), timeout=300)
    assert res.returncode == 0, res.stderr[-3000:]
    got = json.loads(res.stdout.strip().splitlines()[-1])
    assert os.path.samefile(got["file"], os.path.join(ROOT, "lanpaint_b200", "comfy_nodes.py"))
    want = json.load(open(os.path.join(GOLDEN_DIR, "node_unit_answers.json")))
    assert want.keys() == got["answers"].keys()
    for key in want:
        assert got["answers"][key] == want[key], key


def test_package_lists_its_nodes_without_comfyui(tmp_path):
    """reference tests/test_LanPaint.py + __init__.py:90-98: importable, NODE_CLASS_MAPPINGS introspectable, where
    neither ComfyUI nor any stand-in is installed (a clean interpreter, not this test process)."""
    code = (
        "import sys, json\n"
        f"sys.path.insert(0, {ROOT!r})\n"
        "import lanpaint_b200\n"
        "m = lanpaint_b200.NODE_CLASS_MAPPINGS\n"
        "import comfy\n"
        "assert getattr(comfy, '__lanpaint_b200_tooling_stub__', False)\n"
        "sched = json.dumps(comfy.samplers.KSampler.SCHEDULERS)\n"
        "out = {k: json.loads(json.dumps(v.INPUT_TYPES(), ensure_ascii=False).replace(sched, json.dumps(['<SCHEDULERS>'])))"
        " for k, v in m.items()}\n"
        "print(json.dumps({'inputs': out, 'names': lanpaint_b200.NODE_DISPLAY_NAME_MAPPINGS, 'web': lanpaint_b200.WEB_DIRECTORY}))\n")
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=str(tmp_path), timeout=300)
    assert res.returncode == 0, res.stderr[-2000:]
    got = json.loads(res.stdout.strip().splitlines()[-1])
    api = json.load(open(os.path.join(GOLDEN_DIR, "node_api.json")))
    for name in ("LanPaint_KSampler", "LanPaint_KSamplerAdvanced", "LanPaint_SamplerCustom", "LanPaint_SamplerCustomAdvanced"):
        assert got["inputs"][name] == api[name]["INPUT_TYPES"], name
        assert got["names"][name] == api[name]["display_name"]
    assert got["web"] == "./web" and os.path.isdir(os.path.join(ROOT, "lanpaint_b200", "web"))
