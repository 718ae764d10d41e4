"""Exact-window GEMM on wide token boxes: times one inference on a 'plateau' feature video, whose correlation peaks are
flat enough that the arg-maxes of a cell's members spread over several tokens, so most cells need a 21-wide box
(bench.py's video puts nearly every cell in a 16 x 16 box).

  python tools/bench_xw_boxes.py [--steps 10] [--passes 16] [--noise 1.0]

Prints one JSON line: step time (CUDA events), per-kernel-class times of the exact-window pipeline (the library's
CUDA-event classes), and the exact-window statistics of the last call, including its cells by box part count.
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def plateau_features(T, C, device, seed, noise, passes):
    """bench.synth_video_features with the field smoothed `passes` times (and rescaled to unit standard deviation):
    wider correlation peaks, so the members of a cell disagree by a few tokens on their arg-max."""
    g = torch.Generator(device=device).manual_seed(seed)
    pad = 8
    base = torch.randn(C, bench.GEO_H + 2 * pad, bench.GEO_W + 2 * pad, device=device, generator=g)
    for _ in range(passes):
        sm = base.clone()
        sm[:, 1:-1, 1:-1] = base[:, 1:-1, 1:-1] * 0.5 + 0.125 * (base[:, :-2, 1:-1] + base[:, 2:, 1:-1] +
                                                                 base[:, 1:-1, :-2] + base[:, 1:-1, 2:])
        base = sm
    base /= base.std()
    cg = torch.Generator().manual_seed(seed)
    shifts = torch.zeros(T, 2, dtype=torch.long)
    for t in range(1, T):
        shifts[t] = (shifts[t - 1] + torch.randint(-1, 2, (2,), generator=cg)).clamp(-3, 3)
    feats = torch.empty(T, C, bench.GEO_H, bench.GEO_W, device=device)
    for t in range(T):
        dy, dx = int(shifts[t, 0]), int(shifts[t, 1])
        feats[t] = base[:, pad + dy: pad + dy + bench.GEO_H, pad + dx: pad + dx + bench.GEO_W]
        feats[t] += noise * torch.randn(C, bench.GEO_H, bench.GEO_W, device=device, generator=g)
    return feats


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--T", type=int, default=50)
    ap.add_argument("--C", type=int, default=1024)
    ap.add_argument("--nq", type=int, default=256)
    ap.add_argument("--passes", type=int, default=16)
    ap.add_argument("--noise", type=float, default=1.0)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    a = ap.parse_args()
    dev = "cuda:0"
    import __graft_entry__ as ge
    ge.build()
    from dino_tracker_b200 import ModelInference, Tracker, _lib
    from dino_tracker_b200 import model_inference as mim
    lib = _lib.load()
    feats = plateau_features(a.T, a.C, dev, 4321, a.noise, a.passes)
    model = Tracker(video=torch.zeros(a.T, 3, bench.H, bench.W, device=dev), dino_embed_video=feats, device=dev,
                    delta_channels=[3, 4, 4, 4, a.C])
    del feats
    model.tracker_head.load_state_dict(bench.head_weights_for("sharp"))
    mim.DEFAULT_CHUNK_MAPS = 32768
    _lib.check(lib.dinotrk_infer_set_path(1), "infer_set_path")
    mi = ModelInference(model, model.range_normalizer, 0.7, 0.6)
    q = bench.query_lattice(a.nq, 0).to(dev)
    for _ in range(a.warmup):
        mi.infer(q)
    torch.cuda.synchronize()
    stats = _lib.infer_stats()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.steps):
        mi.infer(q)
    e1.record()
    torch.cuda.synchronize()
    step_ms = e0.elapsed_time(e1) / a.steps
    _lib.profile_enable(True)       # per-class times in a pass of their own (the event pairs serialise the streams)
    _lib.profile_collect()
    for _ in range(a.steps):
        mi.infer(q)
    torch.cuda.synchronize()
    prof = _lib.profile_collect()
    _lib.profile_enable(False)
    kernels = {k: v[0] / a.steps for k, v in prof.items() if k.startswith("xw_")}
    print(json.dumps({"workload": f"plateau video (smoothing passes {a.passes}, noise {a.noise}), T={a.T}, C={a.C}, "
                                  f"{a.nq} query points, exact-window pipeline",
                      "device": torch.cuda.get_device_name(0), "step_ms": step_ms,
                      "anchor_xw_ms_per_step": sum(kernels.values()), "kernels_ms_per_step": kernels, "stats": stats}))


if __name__ == "__main__":
    main()
