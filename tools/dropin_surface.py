"""Extracts the attribute surface the reference's own entry points touch on ``Tracker`` / ``ModelInference`` objects and
writes tests/golden/dropin_surface.json (needs the reference tree; ``python -m oracle.make_golden`` records the digest of the
extraction, which the CPU test checks the committed copy against).

Walked (AssafSinger94/dino-tracker @ 5b0f2b0): inference_grid.py, inference_benchmark.py (variables ``model``,
``model_inference``), dino_tracker.py::get_model / train_setup (``model``), models/model_inference.py (``self.model`` /
``model`` inside ModelInference and the module-level helpers -- what a drop-in Tracker must offer to the reference's
ModelInference, and what a drop-in ModelInference must itself provide); and, separately (``trainer_tracker_attributes``),
everything ANY method of dino_tracker.py::DINOTracker touches on ``model`` -- the training loop, its losses and the
cycle-consistency / contrastive helpers (SURVEY 8f-4)."""
import ast
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def attrs_on(tree, names):
    """Attribute names read/called on plain variables in ``names`` or on ``self.<name>``."""
    found = set()
    for node in ast.walk(tree):
        if isinstance(node, ast.Attribute):
            v = node.value
            if isinstance(v, ast.Name) and v.id in names:
                found.add(node.attr)
            elif isinstance(v, ast.Attribute) and isinstance(v.value, ast.Name) and v.value.id == "self" and v.attr in names:
                found.add(node.attr)
    return found


def tracker_kwargs(tree):
    """Keys of the ``tracker_args`` dict dino_tracker.py::get_model passes to Tracker(**tracker_args)."""
    for node in ast.walk(tree):
        if isinstance(node, ast.Assign) and any(isinstance(t, ast.Name) and t.id == "tracker_args" for t in node.targets) \
                and isinstance(node.value, ast.Dict):
            return sorted(k.value for k in node.value.keys if isinstance(k, ast.Constant))
    return []


def surface(ref):
    def parse(rel):
        return ast.parse(open(os.path.join(ref, rel)).read())
    grid, bench, dt, mi = (parse(p) for p in ("inference_grid.py", "inference_benchmark.py", "dino_tracker.py",
                                              os.path.join("models", "model_inference.py")))
    tracker = attrs_on(grid, {"model"}) | attrs_on(bench, {"model"}) | attrs_on(mi, {"model"})
    for node in ast.walk(dt):   # get_model / train_setup only (the training loop is out of scope)
        if isinstance(node, ast.FunctionDef) and node.name in ("get_model", "train_setup"):
            tracker |= attrs_on(node, {"model"})
    trainer = set()
    for node in ast.walk(dt):
        if isinstance(node, ast.ClassDef) and node.name == "DINOTracker":
            trainer |= attrs_on(node, {"model"})
    trainer.discard("module")          # `model.module if hasattr(model, "module")`: DataParallel unwrapping, not a Tracker attribute
    minf = attrs_on(grid, {"model_inference"}) | attrs_on(bench, {"model_inference"})
    mi_kwargs = set()
    for tree in (grid, bench):
        for node in ast.walk(tree):
            if isinstance(node, ast.Call) and isinstance(node.func, ast.Name) and node.func.id == "ModelInference":
                mi_kwargs |= {k.arg for k in node.keywords}
    infer_kwargs = set()
    for tree in (grid, bench):
        for node in ast.walk(tree):
            if isinstance(node, ast.Call) and isinstance(node.func, ast.Attribute) and node.func.attr == "infer":
                infer_kwargs |= {k.arg for k in node.keywords}
    module_funcs = sorted(n.name for n in mi.body if isinstance(n, ast.FunctionDef))
    mi_methods = sorted(n.name for c in mi.body if isinstance(c, ast.ClassDef) and c.name == "ModelInference"
                        for n in c.body if isinstance(n, ast.FunctionDef) and not n.name.startswith("__"))
    return {"tracker_attributes": sorted(tracker), "trainer_tracker_attributes": sorted(trainer),
            "tracker_ctor_kwargs": tracker_kwargs(dt),
            "model_inference_attributes": sorted(minf), "model_inference_ctor_kwargs": sorted(mi_kwargs),
            "infer_kwargs": sorted(infer_kwargs), "model_inference_module_functions": module_funcs,
            "model_inference_methods": mi_methods}


if __name__ == "__main__":
    ref = sys.argv[1] if len(sys.argv) > 1 else "/root/reference"
    out = surface(ref)
    json.dump(out, open(os.path.join(ROOT, "tests", "golden", "dropin_surface.json"), "w"), indent=1)
    print(json.dumps(out, indent=1))
