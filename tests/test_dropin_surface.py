"""CPU: the surface the reference's own entry points touch (inference_grid.py, inference_benchmark.py,
dino_tracker.py::get_model / train_setup, models/model_inference.py) exists on the drop-in classes.  The surface is
extracted from the reference sources by tools/dropin_surface.py (AST walk) and committed as
tests/golden/dropin_surface.json; the digest of that extraction is recorded in tests/golden/reference_digests.json."""
import inspect
import json
import os
import re
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SURFACE = json.load(open(os.path.join(ROOT, "tests", "golden", "dropin_surface.json")))


def _instance_attributes(cls):
    """Names assigned as ``self.<name> = ...`` anywhere in the class source + class-level names (methods, properties)."""
    src = inspect.getsource(cls)
    names = set(re.findall(r"self\.([A-Za-z_][A-Za-z0-9_]*)\s*=", src))
    for c in cls.__mro__:
        names |= set(vars(c).keys())
    return names


def test_surface_fixture_matches_the_reference_tree():
    """The committed surface is the one extracted from the reference's sources (digest recorded from that extraction)."""
    from oracle import make_golden as mg
    digests = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_digests.json")))
    assert mg.surface_digest(SURFACE) == digests["dropin_surface"]


def test_tracker_offers_everything_the_reference_touches():
    from dino_tracker_b200.tracker import Tracker
    have = _instance_attributes(Tracker)
    missing = [a for a in SURFACE["tracker_attributes"] if a not in have]
    assert not missing, missing
    params = inspect.signature(Tracker.__init__).parameters
    assert all(k in params for k in SURFACE["tracker_ctor_kwargs"])
    # positional order of the reference's constructor (models/tracker.py:20-32)
    assert list(params)[1:11] == ["video", "ckpt_path", "dino_embed_path", "dino_patch_size", "stride", "device",
                                  "cyc_n_frames", "cyc_batch_size_per_frame", "cyc_fg_points_ratio", "cyc_thresh"]


def test_tracker_offers_everything_the_reference_trainer_touches():
    """SURVEY 8f-4: every attribute / method dino_tracker.py::DINOTracker (training loop, losses, cycle-consistency and
    contrastive helpers) uses on ``model``."""
    from dino_tracker_b200.tracker import Tracker
    have = _instance_attributes(Tracker)
    missing = [a for a in SURFACE["trainer_tracker_attributes"] if a not in have]
    assert not missing, missing
    assert "get_point_predictions" in have and "get_cycle_consistent_coords" in have      # models/tracker.py:175-262


def test_model_inference_offers_everything_the_reference_touches():
    from dino_tracker_b200 import model_inference as mi
    have = _instance_attributes(mi.ModelInference)
    missing = [a for a in SURFACE["model_inference_attributes"] + SURFACE["model_inference_methods"] if a not in have]
    assert not missing, missing
    params = inspect.signature(mi.ModelInference.__init__).parameters
    assert all(k in params for k in SURFACE["model_inference_ctor_kwargs"])
    assert all(k in inspect.signature(mi.ModelInference.infer).parameters for k in SURFACE["infer_kwargs"])
    for fn in SURFACE["model_inference_module_functions"]:
        assert callable(getattr(mi, fn)), fn
    # the drop-in package re-exports them under the reference's module paths
    sys.path.insert(0, os.path.join(ROOT, "dino_tracker_b200", "dropin"))
    try:
        for m in [k for k in list(sys.modules) if k == "models" or k.startswith("models.")]:
            del sys.modules[m]
        import models.model_inference as dmi
        import models.tracker as dtr
        assert dmi.ModelInference is mi.ModelInference and dtr.Tracker.__name__ == "Tracker"
        for fn in SURFACE["model_inference_module_functions"]:
            assert getattr(dmi, fn) is getattr(mi, fn)
    finally:
        sys.path.pop(0)
        for m in [k for k in list(sys.modules) if k == "models" or k.startswith("models.")]:
            del sys.modules[m]
