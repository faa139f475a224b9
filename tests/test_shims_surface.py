"""The shim packages (shims/network, shims/tools) must serve everything the reference's scripts take from
`network.models_att`, `tools.tools`, `tools.data` and `tools.params_help` (SURVEY 8(b): "train.py, inference.py and
evaluate.py unchanged").  CPU part: every attribute the scripts access on those modules, every keyword they pass, the
constructor kwargs and methods of `cgcnn` and the signatures of the tools / data functions are checked against the
mirrors.  That surface is read from tests/golden/reference_api.json, or parsed (ast) from the reference's own source when
LCN_REFERENCE_DIR names a checkout of it.  The GPU part (tests/test_gpu_scripts.py) executes the scripts' call sequences."""
import ast
import importlib
import inspect
import json
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("LCN_REFERENCE_DIR")
SCRIPTS = ["train.py", "inference.py", "evaluate.py"]
# graph / session plumbing of cgcnn / base_model that has no counterpart without TensorFlow
NOT_APPLICABLE = {"_get_session", "_variable", "remove_checkpoint", "probabilities", "__init__"}


@pytest.fixture(scope="module")
def shim_modules():
    saved_path, saved_mods = list(sys.path), {k: v for k, v in sys.modules.items() if k == "tools" or k.startswith("tools.") or k == "network" or k.startswith("network.")}
    for k in saved_mods:
        del sys.modules[k]
    sys.path.insert(0, os.path.join(ROOT, "shims"))
    try:
        mods = {"models_att": importlib.import_module("network.models_att"), "tools": importlib.import_module("tools.tools"),
                "data": importlib.import_module("tools.data"), "params_help": importlib.import_module("tools.params_help"),
                "filter_hub": importlib.import_module("tools.filter_hub")}
        assert all(os.path.join(ROOT, "shims") in m.__file__ for m in mods.values())
        yield mods
    finally:
        sys.path[:] = saved_path
        for k in [k for k in sys.modules if k == "tools" or k.startswith("tools.") or k == "network" or k.startswith("network.")]:
            del sys.modules[k]
        sys.modules.update(saved_mods)


def _module_uses(src):
    """-> {module name: set of attributes accessed on it}, [(module name, callee, keyword names)]"""
    tree = ast.parse(src)
    local = {}
    for node in ast.walk(tree):
        if isinstance(node, ast.ImportFrom) and node.module in ("tools", "network"):
            for a in node.names:
                local[a.asname or a.name] = a.name
    uses, calls = {v: set() for v in local.values()}, []
    for node in ast.walk(tree):
        if isinstance(node, ast.Attribute) and isinstance(node.value, ast.Name) and node.value.id in local:
            uses[local[node.value.id]].add(node.attr)
        if isinstance(node, ast.Call) and isinstance(node.func, ast.Attribute):
            f = node.func
            if isinstance(f.value, ast.Name) and f.value.id in local:
                calls.append((local[f.value.id], f.attr, [k.arg for k in node.keywords if k.arg]))
    return uses, calls


def _signatures(tree):
    return {n.name: [a.arg for a in n.args.args] for n in tree.body if isinstance(n, ast.FunctionDef)}


def _parse_reference(ref):
    """The surface reference_api.json records, parsed from the reference checkout at `ref`."""
    read = lambda *p: open(os.path.join(ref, *p)).read()
    api = {"scripts": {}}
    for script in SCRIPTS:
        uses, calls = _module_uses(read(script))
        api["scripts"][script] = {"uses": {m: sorted(a) for m, a in uses.items()}, "calls": calls}
    classes = {n.name: n for n in ast.parse(read("network", "models_att.py")).body if isinstance(n, ast.ClassDef)}
    init = next(n for n in classes["cgcnn"].body if isinstance(n, ast.FunctionDef) and n.name == "__init__")
    api["cgcnn_kwargs"] = [a.arg for a in init.args.args if a.arg != "self"]
    api["cgcnn_methods"] = sorted({n.name for c in ("cgcnn", "base_model") for n in classes[c].body
                                   if isinstance(n, ast.FunctionDef)} - NOT_APPLICABLE)
    api["tools_signatures"] = _signatures(ast.parse(read("tools", "tools.py")))
    dtree = ast.parse(read("tools", "data.py"))
    api["data_signatures"] = _signatures(dtree)
    reader = next(n for n in dtree.body if isinstance(n, ast.ClassDef) and n.name == "DataReader")
    api["datareader_signatures"] = {m.name: [a.arg for a in m.args.args] for m in reader.body
                                    if isinstance(m, ast.FunctionDef) and m.name != "__init__"}
    return api


@pytest.fixture(scope="module")
def reference_api():
    if REF:
        return _parse_reference(REF)
    with open(os.path.join(ROOT, "tests", "golden", "reference_api.json")) as f:
        return json.load(f)


@pytest.mark.parametrize("script", SCRIPTS)
def test_every_module_attribute_the_script_uses_exists(shim_modules, reference_api, script):
    uses, calls = reference_api["scripts"][script]["uses"], reference_api["scripts"][script]["calls"]
    assert uses, script
    for mod, attrs in uses.items():
        for a in sorted(attrs):
            assert hasattr(shim_modules[mod], a), f"{script}: {mod}.{a} is missing from the shim"
    for mod, fn, kws in calls:
        target = getattr(shim_modules[mod], fn)
        sig = inspect.signature(target.__init__ if inspect.isclass(target) else target)
        if any(p.kind == p.VAR_KEYWORD for p in sig.parameters.values()):
            continue
        for k in kws:
            assert k in sig.parameters, f"{script}: {mod}.{fn}(... {k}=) is not accepted by the mirror"


def test_cgcnn_accepts_every_constructor_kwarg_and_method_of_the_reference(shim_modules, reference_api):
    """The constructor kwargs (models_att.py:478-506) and the methods of the reference's cgcnn / base_model classes,
    among them the layer / mask API SURVEY 8(b) lists."""
    mirror = shim_modules["models_att"].cgcnn
    sig = inspect.signature(mirror.__init__).parameters
    for k in reference_api["cgcnn_kwargs"]:
        assert k in sig, k
    for name in reference_api["cgcnn_methods"]:
        assert hasattr(mirror, name), f"cgcnn.{name} is missing"
    for name, n_args in (("mask_weights", 1), ("batch_normalization_warp", 3), ("two_linear", 3), ("kaiming", 2),
                         ("loss", 2), ("training", 4), ("_inference_lcn", 1)):
        params = [p for p in inspect.signature(getattr(mirror, name)).parameters.values() if p.name != "self"]
        required = [p for p in params if p.default is p.empty]
        assert len(required) <= n_args <= len(params), (name, [p.name for p in params])
    assert callable(shim_modules["models_att"].get_exponential_matrix)


def test_tools_functions_keep_the_reference_signatures(shim_modules, reference_api):
    ref = reference_api["tools_signatures"]
    for fn in ("procrustes", "image_to_camera_frame", "align_to_gt"):
        got = list(inspect.signature(getattr(shim_modules["tools"], fn)).parameters)
        assert got == ref[fn], (fn, got, ref[fn])
    dref = reference_api["data_signatures"]
    for fn in ("flip_data", "translation_data", "rotate_data", "undo", "get_subset"):
        got = list(inspect.signature(getattr(shim_modules["data"], fn)).parameters)
        assert got == dref[fn], (fn, got, dref[fn])
    for name, args in reference_api["datareader_signatures"].items():
        got = list(inspect.signature(getattr(shim_modules["data"].DataReader, name)).parameters)
        assert got == args, (name, got)


def test_optional_stubs_have_no_arithmetic():
    sys.path.insert(0, os.path.join(ROOT, "shims", "optional_stubs"))
    try:
        for k in ("prettytable",):
            sys.modules.pop(k, None)
        import prettytable
        t = prettytable.PrettyTable()
        t.field_names = ["test_name", 0, "avg"]
        t.add_row(["test1", "12.30", "12.30"])
        assert "12.30" in str(t) and "test_name" in str(t)
    finally:
        sys.path.remove(os.path.join(ROOT, "shims", "optional_stubs"))
        sys.modules.pop("prettytable", None)
