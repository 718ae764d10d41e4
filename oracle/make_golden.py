"""Generate ``tests/golden/*.npz`` by running the LIVE reference modules (build container only).

    python -m oracle.make_golden            # rewrites every fixture

Test infrastructure (see ``oracle/__init__.py``).  Inputs come from ``oracle/synth.py``
(seeded, regenerable); outputs are whatever the unmodified reference code under
``/root/reference`` returns on CPU behind the three shims of ``oracle/ref_harness.py``.
"""
import hashlib
import json
import os
import sys

import numpy as np
import torch

from . import ref_harness, synth
from . import delta_dino as od

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")

# name: geometry / sizes / seeds of every tracker+inference case
TRACK_CASES = {
    "track_small_well":  dict(H=98, W=126, T=6, C=32, seed=11, head="well", nq=(3, 2), tq=[0, 2, 5, 1, 3, 4], batch=None, noise=0.15),
    "track_small_sharp": dict(H=98, W=126, T=6, C=32, seed=12, head="sharp", nq=(3, 2), tq=[0, 2, 5, 1, 3, 4], batch=None, noise=0.15),
    "track_small_chunk": dict(H=98, W=126, T=7, C=32, seed=13, head="well", nq=(2, 2), tq=[0, 6, 3, 2], batch=3, noise=0.15),
    "track_small_fallback": dict(H=98, W=126, T=5, C=32, seed=14, head="default", nq=(2, 2), tq=[0, 1, 2, 4], batch=None, noise=0.15),
    "track_small_mixed": dict(H=98, W=126, T=5, C=32, seed=15, head="mixed", nq=(2, 2), tq=[0, 1, 2, 4], batch=None, noise=0.15),
    "track_small_noisy": dict(H=98, W=126, T=8, C=48, seed=16, head="sharp", nq=(3, 3), tq=[0, 1, 2, 3, 4, 5, 6, 7, 0], batch=None, noise=0.9),
    "track_full_fallback": dict(H=476, W=854, T=3, C=16, seed=18, head="default", nq=(2, 2), tq=[0, 1, 2, 1], batch=None, noise=0.15),
    "track_full_geom":   dict(H=476, W=854, T=4, C=32, seed=17, head="sharp", nq=(2, 2), tq=[0, 1, 2, 3], batch=None, noise=0.15),
}


def case_inputs(cfg):
    """Inputs of a tracker case, regenerable anywhere from the seeds in ``cfg``."""
    from .tracker import Geometry
    geo = Geometry(H=cfg["H"], W=cfg["W"])
    feats, _ = synth.shifted_field_features(cfg["T"], cfg["C"], geo.h, geo.w, seed=cfg["seed"],
                                            noise=cfg["noise"], max_shift=2)
    head = synth.head_weights(cfg["head"], seed=cfg["seed"])
    q = synth.lattice_query_points(cfg["nq"][0], cfg["nq"][1], cfg["H"], cfg["W"], t_q=cfg["tq"],
                                   margin=12.0, jitter_seed=cfg["seed"])
    return geo, feats, head, q


def gen_track_case(name, cfg):
    geo, feats, head, q = case_inputs(cfg)
    T = cfg["T"]
    video = torch.zeros(T, 3, cfg["H"], cfg["W"])
    model = ref_harness.build_reference_tracker(video, feats, head_sd=head,
                                                delta_channels=[3, 2, 2, 2, cfg["C"]])
    from models.model_inference import ModelInference
    from data.dataset import RangeNormalizer
    rn = RangeNormalizer(shapes=(cfg["W"], cfg["H"], T))
    with torch.no_grad():
        mi = ModelInference(model, rn, 0.7, 0.6)
        # default-initialised delta-DINO has an exactly-zero residual (zero last conv, BN(0)=0)
        assert torch.equal(model.refined_features, feats)
        trajs = mi.compute_trajectories(q, cfg["batch"])
        cos = mi.compute_trajectory_cos_sims(trajs, q)
        anch = mi.compute_anchor_trajectories(trajs, cos, cfg["batch"])
        occ = mi.compute_occlusion(trajs, cos, anch)
        traj2, occ2 = mi.infer(q, cfg["batch"])
        assert torch.equal(traj2, trajs[..., :2]) and torch.equal(occ2, occ)
        # one raw forward (normalised output) for the first query point
        from models.model_inference import generate_trajectory_input
        inp = generate_trajectory_input(q[0], model.video)
        fwd = model(inp)
    N = q.shape[0]
    anchors_pad = np.full((N, T, T, 2), np.nan, dtype=np.float32)
    n_anch = np.zeros(N, dtype=np.int64)
    for n in range(N):
        m = anch[n].shape[0]
        n_anch[n] = m
        anchors_pad[n, :m] = anch[n].numpy()
    out = dict(query_points=q.numpy(), trajectories=trajs.numpy(), cos_sims=cos.numpy(),
               anchors=anchors_pad, n_anchors=n_anch, occlusion=occ.numpy(), forward0=fwd.numpy(),
               feat_checksum=np.array([feats.double().sum().item(), feats.double().abs().sum().item()]))
    if feats.numel() * 4 < 400_000:
        out["features"] = feats.numpy()
    for k, v in head.items():
        out["head." + k] = v.numpy()
    np.savez_compressed(os.path.join(GOLDEN_DIR, name + ".npz"), **out)
    print(name, "anchors per query", n_anch.tolist(), "occ frac", occ.float().mean().item())


def gen_delta_case(name, H, W, T, channels, seed):
    g = torch.Generator().manual_seed(seed)
    sd = od.random_state_dict(channels, g, last_std=0.05)
    video = synth.random_video(T, H, W, seed=seed)
    from .tracker import Geometry
    geo = Geometry(H=H, W=W)
    dino = synth.random_features(T, channels[-1], geo.h, geo.w, seed=seed + 1)
    model = ref_harness.build_reference_tracker(video, dino, delta_sd=sd, delta_channels=channels)
    with torch.no_grad():
        model.cache_refined_embeddings()
        refined = model.refined_features
        cnn = video
        for layer in model.delta_dino.layers:
            cnn = layer(cnn)
    out = dict(channels=np.array(channels), seed=np.array(seed), HWT=np.array([H, W, T]))
    ref = refined.numpy()
    if ref.size * 4 < 600_000:
        out["refined"] = ref
        out["cnn_out"] = cnn.numpy()
    else:
        rs = np.random.RandomState(seed)
        idx = rs.randint(0, ref.size, size=4096)
        out["refined_idx"] = idx
        out["refined_vals"] = ref.reshape(-1)[idx]
        out["refined_sum"] = np.array([ref.astype(np.float64).sum(), np.abs(ref.astype(np.float64)).sum()])
    for k, v in sd.items():
        out["sd." + k] = v.numpy()
    np.savez_compressed(os.path.join(GOLDEN_DIR, name + ".npz"), **out)
    print(name, "refined", tuple(refined.shape))


TRAIN_CASE = dict(H=98, W=126, T=6, C=32, channels=[3, 8, 8, 8, 32], seed=51, frames_set=[5, 1, 3, 0], B=48)


def train_case_inputs(cfg=TRAIN_CASE):
    """Inputs of the training-step case (SURVEY 8f-4), regenerable anywhere from the seed."""
    from .tracker import Geometry
    geo = Geometry(H=cfg["H"], W=cfg["W"])
    feats, _ = synth.shifted_field_features(cfg["T"], cfg["C"], geo.h, geo.w, seed=cfg["seed"], noise=0.2, max_shift=2)
    video = synth.random_video(cfg["T"], cfg["H"], cfg["W"], seed=cfg["seed"] + 1)
    head = synth.head_weights("well", seed=cfg["seed"])
    dsd = od.random_state_dict(cfg["channels"], torch.Generator().manual_seed(cfg["seed"] + 2), last_std=0.05)
    g = torch.Generator().manual_seed(cfg["seed"] + 3)
    n_set, B = len(cfg["frames_set"]), cfg["B"]
    pts = torch.rand(B, 3, generator=g) * torch.tensor([cfg["W"] - 1.0, cfg["H"] - 1.0, 0.0])
    src = torch.randint(0, n_set, (B,), generator=g)
    tgt = torch.randint(0, n_set, (B,), generator=g)
    labels = torch.rand(B, 2, generator=g) * 2 - 1
    fs = torch.tensor(cfg["frames_set"], dtype=torch.int64)
    return geo, feats, video, head, dsd, (pts, src, tgt, fs), labels


def train_loss(coords, labels, frame_embeddings, raw_embeddings):
    """The tracking loss of dino_tracker.py:30,411 plus the embedding-norm regulariser of :136-140 (weight 1e-2 here so
    that its gradient is visible next to the tracking term)."""
    huber = torch.nn.HuberLoss(delta=1 / 32, reduction="none")
    reg = (frame_embeddings.norm(dim=1) / raw_embeddings.norm(dim=1) - 1).abs().mean()
    return huber(coords, labels).mean() + 1e-2 * reg


def gen_train_case(name, cfg=TRAIN_CASE):
    """One training-step forward + backward of the LIVE reference in train mode (BatchNorm on batch statistics):
    model(inputs) -> loss -> backward (dino_tracker.py:405-427), gradients of every trainable tensor + of the refined
    embeddings."""
    geo, feats, video, head, dsd, inp, labels = train_case_inputs(cfg)
    model = ref_harness.build_reference_tracker(video, feats, head_sd=head, delta_sd=dsd, delta_channels=cfg["channels"])
    model.train()
    coords = model(inp)
    model.frame_embeddings.retain_grad()
    loss = train_loss(coords, labels, model.frame_embeddings, model.raw_embeddings)
    loss.backward()
    out = dict(coords=coords.detach().numpy(), loss=np.array(loss.item()), grad_frame_embeddings=model.frame_embeddings.grad.numpy())
    for k, p in model.delta_dino.named_parameters():
        out["grad.delta_dino." + k] = p.grad.numpy()
    for k, p in model.tracker_head.named_parameters():
        out["grad.tracker_head." + k] = p.grad.numpy()
    np.savez_compressed(os.path.join(GOLDEN_DIR, name + ".npz"), **out)
    print(name, "loss", loss.item(), "grad norms", {k: float(np.abs(v).max()) for k, v in out.items() if k.startswith("grad")})


CYC_CASE = dict(H=98, W=126, T=6, C=32, seed=61, frames_set=[0, 2, 3, 5], n_frames=3, per_frame=48, fg_ratio=0.7, thresh=20, rng=77)


def cyc_case_inputs(cfg=CYC_CASE):
    """Inputs of the cycle-consistency case (models/tracker.py:182-301)."""
    from .tracker import Geometry
    geo = Geometry(H=cfg["H"], W=cfg["W"])
    feats, _ = synth.shifted_field_features(cfg["T"], cfg["C"], geo.h, geo.w, seed=cfg["seed"], noise=0.1, max_shift=1)
    head = synth.head_weights("sharp", seed=cfg["seed"])
    fg = torch.zeros(cfg["T"], cfg["H"], cfg["W"])
    fg[:, 20:70, 30:100] = 1
    fs = torch.tensor(cfg["frames_set"], dtype=torch.int64)
    g = torch.Generator().manual_seed(cfg["seed"] + 1)
    pts = torch.rand(8, 3, generator=g) * torch.tensor([cfg["W"] - 1.0, cfg["H"] - 1.0, 0.0])
    inp = (pts, torch.randint(0, 4, (8,), generator=g), torch.randint(0, 4, (8,), generator=g), fs)
    return geo, feats, head, fg, inp


def gen_cycle_case(name, cfg=CYC_CASE):
    """``Tracker.get_cycle_consistent_preds`` of the LIVE reference on the CPU (cached refined features = the synthetic
    features: default-initialised delta-DINO has a zero residual), random draws seeded right before the call."""
    geo, feats, head, fg, inp = cyc_case_inputs(cfg)
    model = ref_harness.build_reference_tracker(torch.zeros(cfg["T"], 3, cfg["H"], cfg["W"]), feats, head_sd=head,
                                                delta_channels=[3, 2, 2, 2, cfg["C"]])
    model.cyc_n_frames, model.cyc_batch_size_per_frame = cfg["n_frames"], cfg["per_frame"]
    model.cyc_fg_points_ratio, model.cyc_thresh = cfg["fg_ratio"], cfg["thresh"]
    with torch.no_grad():
        model.cache_refined_embeddings()
        model(inp)                                   # the step's forward: its frame set's embeddings feed the cycle search
        torch.manual_seed(cfg["rng"])
        preds = model.get_cycle_consistent_preds(inp[-1], fg)
    out = {k: v.detach().numpy() for k, v in preds.items()}
    d = out["cycle_consistency_dists"]
    assert d.shape[0] > 20 and d.max() < cfg["thresh"] - 0.5, (d.shape, d.max())     # no survivor near the threshold
    np.savez_compressed(os.path.join(GOLDEN_DIR, name + ".npz"), **out)
    print(name, "survivors", d.shape[0], "of", cfg["n_frames"] * cfg["per_frame"], "max cycle distance", float(d.max()))


def gen_bb_case(name, H, W, T, C, seed):
    import argparse
    import tempfile
    ref_harness.install("cpu")
    from preprocessing_dino_bb import extract_dino_best_buddies as bb
    from .tracker import Geometry
    geo = Geometry(H=H, W=W)
    feats, _ = synth.shifted_field_features(T, C, geo.h, geo.w, seed=seed, noise=0.5, max_shift=2)
    d = tempfile.mkdtemp()
    torch.save(feats, os.path.join(d, "f.pt"))
    args = argparse.Namespace(dino_emb_path=os.path.join(d, "f.pt"), h=H, w=W, stride=7,
                              out_path=os.path.join(d, "out", "bb.pt"))
    bb.run(args)
    res = torch.load(args.out_path)
    out = dict(HWTC=np.array([H, W, T, C]), seed=np.array(seed), features=feats.numpy())
    for k, v in res.items():
        for kk, vv in v.items():
            out[f"{k}.{kk}"] = vv.numpy()
    np.savez_compressed(os.path.join(GOLDEN_DIR, name + ".npz"), **out)
    print(name, {k: v["cos_sims"].shape[0] for k, v in res.items()})


def gen_bb_nms_case(name, H, W, T, C, seed):
    """Live preprocessing_dino_bb/compute_dino_bb_nms.py (compute_bb_nms + compute_max_r over every pair) on the best
    buddies the live extract script finds; the token grid needs >= 400 tokens (torch.topk(k=400))."""
    import argparse
    import tempfile
    ref_harness.install("cpu")
    from preprocessing_dino_bb import compute_dino_bb_nms as nms
    from preprocessing_dino_bb import extract_dino_best_buddies as bb
    from preprocessing_dino_bb.dino_bb_utils import create_meshgrid
    from .tracker import Geometry
    geo = Geometry(H=H, W=W)
    assert geo.P >= 400
    feats, _ = synth.shifted_field_features(T, C, geo.h, geo.w, seed=seed, noise=0.5, max_shift=2)
    d = tempfile.mkdtemp()
    torch.save(feats, os.path.join(d, "f.pt"))
    args = argparse.Namespace(dino_emb_path=os.path.join(d, "f.pt"), h=H, w=W, stride=7, out_path=os.path.join(d, "out", "bb.pt"))
    bb.run(args)
    dino_bb = torch.load(args.out_path)
    coords = create_meshgrid(h=H, w=W, step=7)
    for key in list(dino_bb.keys()):                       # run() of compute_dino_bb_nms.py:85-110 with our geometry's grid
        if dino_bb[key].get("r", None) is not None:
            continue
        sf, tf = (int(x) for x in key.split("_"))
        a = nms.compute_bb_nms(dino_bb[f"{sf}_{tf}"], sf, tf, feats, coords, 7, 50, 0.2)
        b = nms.compute_bb_nms(dino_bb[f"{tf}_{sf}"], tf, sf, feats, coords, 7, 50, 0.2)
        a, b = nms.compute_max_r(a, b)
        dino_bb[key], dino_bb[f"{tf}_{sf}"] = a, b
    out = dict(HWTC=np.array([H, W, T, C]), seed=np.array(seed))
    for k, v in dino_bb.items():
        for kk in ("source_coords", "target_coords", "cos_sims", "peak_affs", "r"):
            out[f"{k}.{kk}"] = v[kk].numpy()
    np.savez_compressed(os.path.join(GOLDEN_DIR, name + ".npz"), **out)
    print(name, {k: (v["r"].shape[0], float(v["r"].max())) for k, v in dino_bb.items()})


def gen_posembed_case(name, cases, dim, n_pos, seed):
    """The reference-owned pieces of the ViT stage (row a1): VitExtractor._fix_pos_enc (models/extractor.py:57-85), the
    position-embedding interpolation for stride-7 overlapping patches, run from the live reference on a seeded table.
    DINOv2 calls it as interpolate_pos_encoding(x, w, h) with (w, h) = x.shape[2:] of the B x 3 x H x W input, i.e.
    w = image HEIGHT and h = image WIDTH."""
    import types
    ref_harness.install("cpu")
    from models.extractor import VitExtractor
    fn = VitExtractor._fix_pos_enc(14, (7, 7))
    g = torch.Generator().manual_seed(seed)
    pos = torch.randn(1, 1 + n_pos * n_pos, dim, generator=g)
    out = dict(dim=np.array(dim), n_pos=np.array(n_pos), seed=np.array(seed), pos_embed=pos.numpy(),
               cases=np.array(cases))
    holder = types.SimpleNamespace(pos_embed=pos)
    for (H, W) in cases:
        n_h, n_w = 1 + (H - 14) // 7, 1 + (W - 14) // 7
        x = torch.zeros(1, 1 + n_h * n_w, dim)
        res = fn(holder, x, H, W)
        assert res.shape == (1, 1 + n_h * n_w, dim)
        out[f"out_{H}x{W}"] = res.numpy()
    np.savez_compressed(os.path.join(GOLDEN_DIR, name + ".npz"), **out)
    print(name, cases)


VIT_CASE = dict(model_name="dinov2_vits14", dim=384, heads=6, depth=2, layer=1, H=98, W=126, T=1, seed=51, std=0.05)


def hf_dinov2_layer(dim, heads, sd, i):
    """Block i of a DINOv2 hub state dict as a ``transformers`` Dinov2Layer: an implementation of the DINOv2 block that is
    independent of oracle/vit.py (also used by tests/test_vit_oracle_cpu.py)."""
    from transformers import Dinov2Config
    from transformers.models.dinov2.modeling_dinov2 import Dinov2Layer
    cfg = Dinov2Config(hidden_size=dim, num_attention_heads=heads, num_hidden_layers=1, mlp_ratio=4, layer_norm_eps=1e-6,
                       hidden_act="gelu", layerscale_value=1.0, use_swiglu_ffn=False, qkv_bias=True,
                       attention_probs_dropout_prob=0.0, hidden_dropout_prob=0.0, drop_path_rate=0.0)
    cfg._attn_implementation = "eager"
    layer = Dinov2Layer(cfg).eval()
    p = f"blocks.{i}."
    qkv_w, qkv_b = sd[p + "attn.qkv.weight"], sd[p + "attn.qkv.bias"]
    mapped = {
        "norm1.weight": sd[p + "norm1.weight"], "norm1.bias": sd[p + "norm1.bias"],
        "norm2.weight": sd[p + "norm2.weight"], "norm2.bias": sd[p + "norm2.bias"],
        "attention.attention.query.weight": qkv_w[:dim], "attention.attention.query.bias": qkv_b[:dim],
        "attention.attention.key.weight": qkv_w[dim:2 * dim], "attention.attention.key.bias": qkv_b[dim:2 * dim],
        "attention.attention.value.weight": qkv_w[2 * dim:], "attention.attention.value.bias": qkv_b[2 * dim:],
        "attention.output.dense.weight": sd[p + "attn.proj.weight"], "attention.output.dense.bias": sd[p + "attn.proj.bias"],
        "layer_scale1.lambda1": sd[p + "ls1.gamma"], "layer_scale2.lambda1": sd[p + "ls2.gamma"],
        "mlp.fc1.weight": sd[p + "mlp.fc1.weight"], "mlp.fc1.bias": sd[p + "mlp.fc1.bias"],
        "mlp.fc2.weight": sd[p + "mlp.fc2.weight"], "mlp.fc2.bias": sd[p + "mlp.fc2.bias"],
    }
    assert set(mapped) == set(layer.state_dict())
    layer.load_state_dict(mapped)
    return layer


def vit_case_state_dict(cfg=VIT_CASE):
    from . import vit as ovit
    g = torch.Generator().manual_seed(cfg["seed"])
    sd = ovit.random_state_dict(cfg["depth"], cfg["dim"], g, n_pos=37, std=cfg["std"])
    for i in range(cfg["depth"]):   # LayerScale away from 1 so that its placement matters
        sd[f"blocks.{i}.ls1.gamma"] = 0.5 + torch.rand(cfg["dim"], generator=g)
        sd[f"blocks.{i}.ls2.gamma"] = 0.5 + torch.rand(cfg["dim"], generator=g)
    return sd


def gen_vit_case(name, cfg=VIT_CASE):
    """Row a1 through the LIVE reference: utils.get_dino_features_video + models/extractor.VitExtractor (ImageNet
    normalisation, stride-7 re-striding of the patch convolution, _fix_pos_enc, block hooks, tap point, cls drop,
    rearrange) run unmodified; only ``torch.hub.load`` -- the network download of facebookresearch/dinov2 -- is replaced by
    a stand-in with the DinoVisionTransformer surface the extractor touches (patch_embed.proj, cls_token, pos_embed,
    interpolate_pos_encoding, blocks[i] with .attn.qkv / .attn.attn_drop hook points, forward = prepare tokens + blocks),
    whose blocks are ``transformers``' Dinov2Layer (independent of oracle/vit.py) carrying seeded weights."""
    import torch.nn as nn
    ref_harness.install("cpu")
    import utils as ref_utils
    sd = vit_case_state_dict(cfg)
    dim, heads = cfg["dim"], cfg["heads"]

    class Block(nn.Module):
        def __init__(self, i):
            super().__init__()
            self.layer = hf_dinov2_layer(dim, heads, sd, i)
            self.attn = nn.Module()                       # hook points only (the extractor registers, never reads, them)
            self.attn.qkv = nn.Identity()
            self.attn.attn_drop = nn.Identity()

        def forward(self, x):
            out = self.layer(x)
            return out[0] if isinstance(out, (tuple, list)) else out

    class StandIn(nn.Module):
        def __init__(self):
            super().__init__()
            self.patch_embed = nn.Module()
            self.patch_embed.proj = nn.Conv2d(3, dim, 14, stride=14)
            self.patch_embed.proj.weight.data.copy_(sd["patch_embed.proj.weight"])
            self.patch_embed.proj.bias.data.copy_(sd["patch_embed.proj.bias"])
            self.cls_token = nn.Parameter(sd["cls_token"].clone())
            self.pos_embed = nn.Parameter(sd["pos_embed"].clone())
            self.blocks = nn.ModuleList([Block(i) for i in range(cfg["depth"])])

        def interpolate_pos_encoding(self, x, w, h):      # replaced by the reference (set_overlapping_patches)
            raise AssertionError("the reference must install its own position-embedding interpolation")

        def forward(self, x):                             # DinoVisionTransformer.prepare_tokens_with_masks + blocks
            B, nc, w, h = x.shape
            x = self.patch_embed.proj(x).flatten(2).transpose(1, 2)
            x = torch.cat((self.cls_token.expand(B, -1, -1), x), dim=1)
            x = x + self.interpolate_pos_encoding(x, w, h)
            for blk in self.blocks:
                x = blk(x)
            return x

    video = synth.random_video(cfg["T"], cfg["H"], cfg["W"], seed=cfg["seed"] + 1)
    real_load = torch.hub.load
    torch.hub.load = lambda repo, model_name, *a, **kw: StandIn().eval()
    try:
        with torch.no_grad():
            feats = ref_utils.get_dino_features_video(video, model_name=cfg["model_name"], stride=7, layer=cfg["layer"],
                                                      device="cpu")
    finally:
        torch.hub.load = real_load
    out = dict(features=feats.numpy(), shape=np.array(feats.shape))
    np.savez_compressed(os.path.join(GOLDEN_DIR, name + ".npz"), **out)
    print(name, tuple(feats.shape), float(feats.abs().max()))


def train_case_arrays(cfg=TRAIN_CASE):
    """Every input ``gen_train_case`` gives the reference, by name."""
    geo, feats, video, head, dsd, (pts, src, tgt, fs), labels = train_case_inputs(cfg)
    out = dict(features=feats, video=video, points=pts, source_frames=src, target_frames=tgt, frames_set=fs, labels=labels)
    out.update({"head." + k: v for k, v in head.items()})
    out.update({"delta_dino." + k: v for k, v in dsd.items()})
    return {k: v.numpy() for k, v in out.items()}


def cycle_case_arrays(cfg=CYC_CASE):
    """Every input ``gen_cycle_case`` gives the reference, by name."""
    geo, feats, head, fg, (pts, src, tgt, fs) = cyc_case_inputs(cfg)
    out = dict(features=feats, foreground=fg, points=pts, source_frames=src, target_frames=tgt, frames_set=fs)
    out.update({"head." + k: v for k, v in head.items()})
    return {k: v.numpy() for k, v in out.items()}


def array_digest(a):
    """sha256 of an array's dtype, shape and bytes: equal digests = bit-identical arrays."""
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(f"{a.dtype.str} {a.shape} ".encode())
    h.update(a.tobytes())
    return h.hexdigest()


def surface_digest(surface):
    """sha256 of the drop-in surface (tools/dropin_surface.py) in a canonical JSON form."""
    return hashlib.sha256(json.dumps(surface, sort_keys=True).encode()).hexdigest()


def reference_digests(golden_dir=GOLDEN_DIR):
    """What the CPU suite checks without the reference (tests/test_golden_regen_cpu.py, tests/test_dropin_surface.py):
    digests of the inputs the training-step and cycle-consistency cases give the reference and of the fixtures in
    ``golden_dir`` that it returned for them, and the digest of the drop-in surface extracted from the reference's
    sources.  Run right after those fixtures were generated."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("dropin_surface", os.path.join(ROOT, "tools", "dropin_surface.py"))
    tool = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(tool)
    out = {"dropin_surface": surface_digest(tool.surface(ref_harness.REFERENCE_ROOT))}
    for name, inputs in (("train_small", train_case_arrays()), ("cycle_small", cycle_case_arrays())):
        fixture = np.load(os.path.join(golden_dir, name + ".npz"))
        out[name] = {"inputs": {k: array_digest(v) for k, v in sorted(inputs.items())},
                     "outputs": {k: array_digest(fixture[k]) for k in sorted(fixture.files)}}
    return out


def main():
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    torch.set_num_threads(8)
    for name, cfg in TRACK_CASES.items():
        gen_track_case(name, cfg)
    gen_delta_case("delta_small", 98, 126, 3, [3, 8, 12, 16, 24], seed=21)
    gen_delta_case("delta_full_geom", 476, 854, 1, [3, 4, 4, 4, 8], seed=22)
    gen_bb_case("bb_small", 98, 126, 3, 16, seed=31)
    gen_bb_nms_case("bb_nms_small", 154, 210, 3, 16, seed=32)
    gen_posembed_case("posembed", [(476, 854), (98, 126), (112, 140), (518, 518)], dim=6, n_pos=37, seed=41)
    gen_vit_case("vit_small")
    gen_train_case("train_small")
    gen_cycle_case("cycle_small")
    with open(os.path.join(GOLDEN_DIR, "reference_digests.json"), "w") as f:
        json.dump(reference_digests(), f, indent=1)


if __name__ == "__main__":
    main()
