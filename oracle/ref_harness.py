"""Import the *live* reference (``/root/reference``) behind three in-memory shims.

Test infrastructure (see ``oracle/__init__.py``).  Usable only where
``/root/reference`` exists (the build container); never on the GPU box.  Used by
``oracle/make_golden.py`` to produce ``tests/golden/*`` (the fixtures and the
digests that pin them, ``reference_digests.json``).

Shims (SURVEY.md 8c) -- none of them touches the arithmetic of the hot path:
  1. ``antialiased_cnns.BlurPool`` (third-party, adobe/antialiased-cnns, not
     vendored, not installed): restated from its published default
     (filt_size=4 -> outer([1,3,3,1])/64, reflect pad (1,2,1,2), stride 2,
     depthwise, buffer ``filt`` of shape C x 1 x 4 x 4); used by
     ``models/networks/delta_dino.py:44``.
  2. ``data.dataset.RangeNormalizer.__init__`` has ``device='cuda'`` as default
     (``data/dataset.py:15``) and is constructed without a device in
     ``models/tracker.py:62`` and ``models/networks/tracker_head.py:112``; the
     default is patched to the harness device.
  3. empty stub modules for ``imageio`` / ``matplotlib`` so that
     ``data/data_utils.py`` imports.
"""
import os
import sys
import types

import torch
import torch.nn as nn
import torch.nn.functional as F

REFERENCE_ROOT = os.environ.get("DINOTRK_REFERENCE_ROOT", "/root/reference")
_installed = {"done": False, "device": None}


def reference_available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "models", "tracker.py"))


class _BlurPool(nn.Module):
    def __init__(self, channels, pad_type="reflect", filt_size=4, stride=2, pad_off=0):
        super().__init__()
        assert filt_size == 4 and pad_type == "reflect" and pad_off == 0
        a = torch.tensor([1.0, 3.0, 3.0, 1.0])
        filt = a[:, None] * a[None, :]
        filt = filt / filt.sum()
        self.register_buffer("filt", filt[None, None].repeat(channels, 1, 1, 1))
        self.stride = stride
        self.channels = channels

    def forward(self, x):
        x = F.pad(x, (1, 2, 1, 2), mode="reflect")
        return F.conv2d(x, self.filt, stride=self.stride, groups=self.channels)


def install(device: str = "cpu") -> None:
    """Put the reference on sys.path behind the shims (idempotent)."""
    if not reference_available():
        raise RuntimeError(f"reference not found at {REFERENCE_ROOT}")
    if _installed["done"]:
        if _installed["device"] != device:
            import data.dataset as ds
            ds.RangeNormalizer._harness_device = device
            _installed["device"] = device
        return
    m = types.ModuleType("antialiased_cnns")
    m.BlurPool = _BlurPool
    sys.modules.setdefault("antialiased_cnns", m)
    for name in ("imageio", "imageio.v3", "matplotlib", "matplotlib.pyplot"):
        sys.modules.setdefault(name, types.ModuleType(name))
    # the reference root must win over any same-named package (our drop-in "models")
    for k in [k for k in sys.modules if k == "models" or k.startswith("models.")
              or k == "data" or k.startswith("data.") or k == "utils"]:
        del sys.modules[k]
    sys.path.insert(0, REFERENCE_ROOT)
    import data.dataset as ds

    orig_init = ds.RangeNormalizer.__init__
    ds.RangeNormalizer._harness_device = device

    def patched_init(self, shapes, device=None):
        orig_init(self, shapes, device=device or ds.RangeNormalizer._harness_device)

    ds.RangeNormalizer.__init__ = patched_init
    _installed["done"] = True
    _installed["device"] = device


def build_reference_tracker(video, dino_features, head_sd=None, delta_sd=None,
                            delta_channels=None, device="cpu", workdir=None,
                            patch_size=14, stride=7):
    """Construct the reference ``models.tracker.Tracker`` on synthetic data.

    video: T x 3 x H x W in [0,1]; dino_features: T x C x h x w.
    ``delta_channels`` lets small tests shrink the CNN (the reference hard-codes
    [3,64,128,256,1024], ``models/networks/delta_dino.py:9``).
    """
    import tempfile
    install(device)
    import models.networks.delta_dino as dd
    from models.tracker import Tracker

    workdir = workdir or tempfile.mkdtemp(prefix="dinotrk_ref_")
    path = os.path.join(workdir, "dino_embed_video.pt")
    torch.save(dino_features.clone(), path)
    orig = dd.DeltaDINO.__init__
    if delta_channels is not None:
        def init(self, *a, **kw):
            kw.setdefault("channels", list(delta_channels))
            orig(self, *a, **kw)
        dd.DeltaDINO.__init__ = init
    try:
        model = Tracker(video=video.to(device), ckpt_path=workdir, dino_embed_path=path,
                        dino_patch_size=patch_size, stride=stride, device=device)
    finally:
        dd.DeltaDINO.__init__ = orig
    if head_sd is not None:
        model.tracker_head.load_state_dict(head_sd)
    if delta_sd is not None:
        model.delta_dino.load_state_dict(delta_sd)
    return model.to(device).eval()
