#!/usr/bin/env python
"""bench.py -- query-points/sec of the DINO-Tracker inference hot path on B200 (BASELINE.json metric).

One "step" = one ``ModelInference.infer`` over one synthetic 854x476, T=50 video with 256 query points
(BASELINE.json configs[1]): trajectories, cos-sims, anchor re-tracking, occlusion.  1 query-point = one
row of ``infer`` output (T-frame trajectory + T-frame occlusion mask), SURVEY.md 8d.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

* ``value``  : whole-job query-points/s, inputs resident in HBM, device-timed (CUDA events), max over ranks.
* ``e2e``    : same metric through the public API with HOST buffers: pinned query points H2D, result D2H
               inside the timed region.
* ``roofline``: dominant kernel of the step (per-kernel CUDA-event times recorded inside the timed region).
* ``cpu_baseline`` / ``--impl reference``: the oracle's faithful restatement of the reference's PyTorch
  path (same einsum / gathers per model() call) on the host cores, on a bounded sample of the workload.

N > 1 (torchrun, one rank per GPU): video-parallel -- every rank tracks its own video of the same shape
(BASELINE configs[2] style), no data-path collective; weak scaling.

``--dump-outputs DIR`` writes what ``infer`` returned in the last timed step (rank 0) as ``DIR/trajectories.npy``
(N x T x 2 px, float32) and ``DIR/occlusion.npy`` (N x T, float32 0 / 1).  The inputs are seeded, so two builds run with
the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark leaves the source tree as it found it (it may be read-only)

H, W = 476, 854
GEO_H, GEO_W = 67, 121
P = GEO_H * GEO_W


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--T", type=int, default=50)
    ap.add_argument("--C", type=int, default=1024, help="feature dim: 1024 = ViT-L/14@15 (shipped config), 768 = ViT-B/14")
    ap.add_argument("--nq", type=int, default=256)
    ap.add_argument("--noise", type=float, default=0.25)
    ap.add_argument("--chunk-maps", type=int, default=32768)
    ap.add_argument("--precision", default="fp16x3", choices=["fp16x3", "fp32"],
                    help="wide correlation groups: tcgen05 3xTF32 tensor cores, or the exact-fp32 FFMA GEMM")
    ap.add_argument("--cpu-baseline", type=int, default=1, help="0: skip the cpu_baseline leg")
    ap.add_argument("--stream-probe", type=int, default=1, help="0: skip the dedicated corr_stream HBM probe")
    ap.add_argument("--stages", type=int, default=1, help="0: skip the ViT / delta-DINO / best-buddies stage timings")
    ap.add_argument("--head", default="sharp", choices=["sharp", "well", "mixed"], help="refiner weights of the timed step")
    ap.add_argument("--path", type=int, default=-1, help="anchor-phase pipeline: -1 automatic, 0 full-map, 1 coarse pass + exact window")
    ap.add_argument("--torch-cuda-baseline", type=int, default=1, help="0: skip timing the reference's PyTorch path on cuda:0")
    ap.add_argument("--second-head", type=int, default=1, help="0: skip the extra timing with the mixed-sign head")
    ap.add_argument("--multi", type=int, default=1, help="0: skip the config 3 / 4 / 5 blocks (bench_multi.py)")
    ap.add_argument("--config3-vit", type=int, default=1, help="0: config 3 without the ViT stage (tracker + delta-DINO only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy (--impl b200)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    return args


def synth_video_features(T, C, device, seed, noise):
    """Shifted smooth descriptor field + per-frame noise (same construction as oracle/synth.py, drawn with
    torch's generator on the target device so that 1.7 GB of features need no host pass)."""
    g = torch.Generator(device=device).manual_seed(seed)
    pad = 8
    base = torch.randn(C, GEO_H + 2 * pad, GEO_W + 2 * pad, device=device, generator=g)
    sm = base.clone()
    sm[:, 1:-1, 1:-1] = base[:, 1:-1, 1:-1] * 0.5 + 0.125 * (base[:, :-2, 1:-1] + base[:, 2:, 1:-1] +
                                                             base[:, 1:-1, :-2] + base[:, 1:-1, 2:])
    cg = torch.Generator().manual_seed(seed)
    shifts = torch.zeros(T, 2, dtype=torch.long)
    for t in range(1, T):
        shifts[t] = (shifts[t - 1] + torch.randint(-1, 2, (2,), generator=cg)).clamp(-3, 3)
    feats = torch.empty(T, C, GEO_H, GEO_W, device=device)
    for t in range(T):
        dy, dx = int(shifts[t, 0]), int(shifts[t, 1])
        feats[t] = sm[:, pad + dy: pad + dy + GEO_H, pad + dx: pad + dx + GEO_W]
        feats[t] += noise * torch.randn(C, GEO_H, GEO_W, device=device, generator=g)
    return feats


def query_lattice(nq, seed):
    side = int(round(nq ** 0.5))
    assert side * side == nq, "--nq must be a square number"
    from bench_inputs import lattice  # not the oracle: the product arm never imports it
    return lattice(side, side, H, W, 0, 30.0, seed)


class ClockSampler:
    """SM clock and clock-event (throttle) reasons sampled DURING the timed region (B200_PROFILING.md's clocks line):
    NVML from a Python thread every 20 ms; `nvidia-smi -lms` as the fallback when pynvml is missing."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
            0x80: "hw_power_brake_slowdown"}

    def __init__(self, index):
        self.index, self.rows, self.proc, self.nvml, self.stop_flag = index, [], None, None, False

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nvml = pynvml
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, bufsize=1)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _poll(self):
        n = self.nvml
        mx = n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)
        while not self.stop_flag:
            try:
                sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
                try:
                    bits = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                except Exception:
                    bits = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                self.rows.append((time.perf_counter(), float(sm), float(mx), int(bits)))
            except Exception:
                pass
            time.sleep(0.02)

    def _read(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.strip().split(",")]
            try:
                bits = 0
                for b, name in zip((0x8, 0x40, 0x20, 0x4), f[3:7]):
                    if name.lower().startswith("active"):
                        bits |= b
                self.rows.append((time.perf_counter(), float(f[0]), float(f[1]), bits))
            except Exception:
                continue

    def stop(self, t0, t1):
        if self.nvml is None and self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no NVML / nvidia-smi"], "samples": 0}
        time.sleep(0.1)
        self.stop_flag = True
        if self.proc is not None:
            self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ts, s_, m_, bits in self.rows:
            if not (t0 <= ts <= t1):
                continue
            sm.append(s_); mx.append(m_)
            for b, name in self.BITS.items():
                if bits & b:
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvml" if self.nvml else "nvidia-smi"}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tf_burst": d["bf16_tflops"], "tf_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "which": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "which": "fallback (B200_PROFILING.md)"}


# ------------------------------------------------------------------------------------------ reference arm
_CPU_FEATS = {}


def head_weights_for(kind):
    """Refiner weights of the timed step: 'sharp' (bench_inputs.sharp_head: positive, dominant centre tap -- like a trained
    head), 'well' (U(0.2, 1) everywhere: blurry softmax) or 'mixed' (mixed-sign kernels).  Same draws as oracle/synth.py."""
    from bench_inputs import sharp_head
    import numpy as np
    if kind == "sharp":
        return sharp_head(0)
    rs = np.random.RandomState(1000)

    def u(lo, hi, *shape):
        return torch.from_numpy(rs.uniform(lo, hi, size=shape).astype(np.float32))
    if kind == "well":
        return {"cnn_refiner.0.weight": u(0.2, 1, 16, 1, 3, 3), "cnn_refiner.0.bias": u(0.2, 1, 16),
                "cnn_refiner.2.weight": u(0.2, 1, 1, 16, 3, 3), "cnn_refiner.2.bias": u(0.2, 1, 1)}
    w1 = u(-0.5, 1, 16, 1, 3, 3); w2 = u(-0.5, 1, 1, 16, 3, 3)
    return {"cnn_refiner.0.weight": w1, "cnn_refiner.0.bias": u(-0.2, 0.2, 16),
            "cnn_refiner.2.weight": w2, "cnn_refiner.2.bias": u(-0.2, 0.2, 1)}


def cpu_reference_sample(T, C, nq, noise, seed=0, anchor_calls=3, samples=3):
    """Times the oracle's FAITHFUL restatement of the reference path (same gathers and B x N einsum per model() call,
    models/tracker.py:303-325) on the host cores, on a bounded sample of the workload: one query point -- per sample its
    trajectory model() call and ``anchor_calls`` anchor model() calls (one untimed warm-up call first), plus the cos-sim
    pass and the occlusion step once.  A query point costs  traj + cos + (#anchors) x anchor-call + occlusion; the value
    uses the MEDIAN call times over ``samples`` samples, the spread (min .. max over samples) is reported next to it.
    Returns (query-points/s, cores, description, seconds per query point, spread dict)."""
    from oracle import inference as oi
    from oracle.tracker import Geometry
    from bench_inputs import sharp_head
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    geo = Geometry()
    key = (T, C, seed, noise)
    if key not in _CPU_FEATS:
        _CPU_FEATS[key] = synth_video_features(T, C, "cpu", seed, noise)
    feats = _CPU_FEATS[key]
    head = sharp_head(0)
    q = query_lattice(nq, seed)[nq // 2 + 3: nq // 2 + 4].clone()
    with torch.no_grad():
        traj = oi.compute_trajectories(feats, q, head, geo, None, faithful=True)          # warm-up (+ the values we need)
        t0 = time.perf_counter()
        cos = oi.compute_trajectory_cos_sims(feats, traj, q, geo)
        t_b = time.perf_counter() - t0
        anchors = torch.arange(T)[cos[0] >= 0.7]
        m = int(anchors.numel())
        k = max(1, min(m, anchor_calls))
        t_traj, t_anchor = [], []
        part = None
        for s_ in range(samples):
            t0 = time.perf_counter()
            oi.compute_trajectories(feats, q, head, geo, None, faithful=True)
            t_traj.append(time.perf_counter() - t0)
            sel = anchors[(torch.arange(k) + s_ * k) % max(m, 1)] if m else anchors
            t0 = time.perf_counter()
            part = oi.anchor_predictions(feats, traj[0], sel, head, geo, None, faithful=True)
            t_anchor.append((time.perf_counter() - t0) / max(len(sel), 1))
        t0 = time.perf_counter()
        green = part.repeat((m + k - 1) // k, 1, 1)[:m] if m else part
        oi.occlusion_for_query(green, traj[0, :, :2], cos[0], 0.7, 0.6)
        t_d = time.perf_counter() - t0
    per_qp = [t_traj[i] + t_b + m * t_anchor[i] + t_d for i in range(samples)]
    total = statistics.median(per_qp)
    spread = {"samples": samples, "anchor_calls_per_sample": k, "s_per_query_point_min": min(per_qp),
              "s_per_query_point_median": total, "s_per_query_point_max": max(per_qp),
              "traj_call_s_median": statistics.median(t_traj), "anchor_call_s_median": statistics.median(t_anchor)}
    desc = (f"1 query point of the T={T}, C={C} workload on {cores} host threads: median over {samples} samples of "
            f"[trajectory model() call {statistics.median(t_traj):.2f}s + {k} anchor model() calls "
            f"{statistics.median(t_anchor):.2f}s each, extrapolated to this point's {m} anchors] + cos-sims {t_b:.2f}s + "
            f"occlusion {t_d:.3f}s; per-query-point seconds min/median/max = {min(per_qp):.1f}/{total:.1f}/{max(per_qp):.1f}")
    return 1.0 / total, cores, desc, total, spread


def torch_cuda_reference_sample(T, C, nq, noise, dev, n_points=2):
    """The reference's PyTorch path on THIS GPU (the north star's >= 10x comparator, SURVEY.md 8d): the oracle's faithful
    restatement (per model() call: two gathered copies of the frame set, B x N einsum, refiner convolutions, softmax --
    models/tracker.py:303-325, models/model_inference.py:37-216) run by torch on ``dev`` with torch's default precision
    flags (fp32 matmul; cuDNN convolutions may use TF32, as they would for the reference), for ``n_points`` complete query
    points (trajectory, cos-sims, every anchor call, occlusion) after one warm-up point."""
    from oracle import inference as oi
    from oracle.tracker import Geometry
    from bench_inputs import sharp_head
    geo = Geometry()
    feats = synth_video_features(T, C, dev, 1234, noise)
    head = {k: v.to(dev) for k, v in sharp_head(0).items()}
    q_all = query_lattice(nq, 0).to(dev)
    idx = [nq // 2 + 3, 5, nq - 7, nq // 3][: n_points + 1]
    with torch.no_grad():
        oi.infer(feats, q_all[idx[:1]], head, geo, 0.7, 0.6, faithful=True)            # warm-up: cuBLAS / cuDNN plans
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        _, _, aux = oi.infer(feats, q_all[idx[1:]], head, geo, 0.7, 0.6, faithful=True, return_all=True)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
    n = len(idx) - 1
    calls = n + int(sum(int(a.shape[0]) for a in aux["anchors"].values()))
    del feats
    torch.cuda.empty_cache()
    return {"value": n / dt, "unit": "query-points/s", "device": torch.cuda.get_device_name(0), "kind": "port",
            "sample": (f"{n} complete query points of the T={T}, C={C} workload ({calls} model() calls, {dt / calls * 1e3:.1f} ms each), "
                       f"the oracle's faithful restatement of the reference path run by torch {torch.__version__} on the GPU, "
                       f"fp32, after one warm-up point"),
            "s_per_query_point": dt / n}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # every step is one bounded sample (~15 s of host time at T=50, C=1024); the whole arm is kept within ~4 minutes:
    # with large --steps only as many samples as fit are measured, and the line reports how many
    vals, descs, budget_s, t_start = [], None, 240.0, time.perf_counter()
    warm = min(args.warmup, 1)
    for i in range(warm + args.steps):
        t_s = time.perf_counter()
        v, cores, desc, total, _ = cpu_reference_sample(args.T, args.C, args.nq, args.noise, seed=0, anchor_calls=1, samples=1)
        dt = time.perf_counter() - t_s
        if i >= warm:
            vals.append(v)
        descs = desc
        if vals and time.perf_counter() - t_start + dt > budget_s:
            break
    value = statistics.mean(vals) if vals else 0.0
    line = {"impl": "reference", "metric": "query-points/sec (854x476, T=%d)" % args.T, "value": value,
            "unit": "query-points/s", "n_gpus": args.gpus, "steps": len(vals), "warmup": warm,
            "steps_requested": args.steps, "warmup_requested": args.warmup,
            "ms_per_step": 1000.0 / value if value else None, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(args), "T": args.T, "C": args.C, "query_points": args.nq},
            "cpu_baseline": {"value": value, "unit": "query-points/s", "cores": cores, "kind": "port", "sample": descs},
            "e2e": {"value": value, "unit": "query-points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def workload_name(args):
    return (f"TAP-Vid-DAVIS-shape single video 854x476, T={args.T}, {args.nq} query points (16x16 lattice, t_q=0), "
            f"C={args.C} ({'ViT-L/14@15' if args.C == 1024 else 'ViT-B/14' if args.C == 768 else 'custom'} features), "
            f"shifted-field synthetic features (noise {args.noise}), refined features cached in HBM")


# ------------------------------------------------------------------------------------------ product arm
DUMP_BYTES = 60_000_000   # array bytes of one dump: with the .npy headers, under 64 MB


def dump_outputs(out_dir, outputs):
    """``outputs``: {name: tensor with one row per query point} -> out_dir/<name>.npy in float32.  Above DUMP_BYTES in all,
    a fixed seeded sample of the rows (ascending) is written instead, with its row indices as query_rows.npy."""
    import numpy as np
    rows = next(iter(outputs.values())).shape[0]
    row_bytes = sum(4 * t[0].numel() for t in outputs.values())
    if rows * row_bytes > DUMP_BYTES:
        keep = torch.randperm(rows, generator=torch.Generator().manual_seed(0))[:DUMP_BYTES // (row_bytes + 4)].sort().values
        outputs = {k: t[keep.to(t.device)] for k, t in outputs.items()}
        outputs["query_rows"] = keep
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def run_b200(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device(dev))

    import __graft_entry__ as ge
    if rank == 0:
        ge.build()
    if dist is not None:
        dist.barrier()
    from dino_tracker_b200 import ModelInference, Tracker, _lib
    lib = _lib.load()

    T, C, nq = args.T, args.C, args.nq
    feats = synth_video_features(T, C, dev, 1234 + rank, args.noise)
    video = torch.zeros(T, 3, H, W, device=dev)  # frames only feed delta-DINO (default init: zero residual)
    model = Tracker(video=video, dino_embed_video=feats, device=dev, delta_channels=[3, 4, 4, 4, C],
                    corr_precision=args.precision)
    del feats
    model.tracker_head.load_state_dict(head_weights_for(args.head))
    from dino_tracker_b200 import model_inference as _mi_mod
    _mi_mod.DEFAULT_CHUNK_MAPS = args.chunk_maps
    _lib.check(lib.dinotrk_infer_set_path(args.path), "infer_set_path")
    mi = ModelInference(model, model.range_normalizer, 0.7, 0.6)
    q_host = query_lattice(nq, 0).pin_memory()
    q_dev = q_host.to(dev)

    def step_resident():
        return mi.infer(q_dev)

    for _ in range(args.warmup):
        step_resident()
    torch.cuda.synchronize()

    # workload facts (anchors per query) from one un-timed call
    r = mi.infer_all(q_dev)
    n_anch = (r["cos_sims"] >= 0.7).sum(dim=1).float()
    maps_per_step = int(nq * T + n_anch.sum().item() * T)
    torch.cuda.synchronize()
    path_stats = _lib.infer_stats()

    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.1)
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    _lib.profile_enable(True)
    _lib.profile_collect()
    launches0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.perf_counter()
    e0.record()
    for _ in range(args.steps):
        last = step_resident()
    e1.record()
    torch.cuda.synchronize()
    t_wall1 = time.perf_counter()
    if dist is not None:
        dist.barrier()
    ms = e0.elapsed_time(e1)
    launches = _lib.launch_count() - launches0
    prof = _lib.profile_collect()
    _lib.profile_enable(False)
    clocks = sampler.stop(t_wall0, t_wall1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"trajectories": last[0], "occlusion": last[1]})

    # ---- e2e: host buffers, H2D + D2H inside the timed region
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        qd = q_host.to(dev, non_blocking=True)
        traj, occ = mi.infer(qd)
        traj_h, occ_h = traj.cpu(), occ.cpu()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    h2d = q_host.numel() * 4
    d2h = traj_h.numel() * 4 + occ_h.numel()

    if dist is not None:
        tt = torch.tensor([ms, e2e_s * 1000.0], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms, e2e_ms = tt[0].item(), tt[1].item()
    else:
        e2e_ms = e2e_s * 1000.0
    # ---- BASELINE configs 3 / 4 / 5 (every rank takes part; rank 0 keeps the blocks)
    multi_blocks = {}
    if args.multi and C == 1024:
        import bench_multi
        import bench as _self
        c_map = (ms / args.steps / 1e3) / float(nq * T * (T + 1))
        mi_keep, model_keep = mi, model
        for name, fn in (("config4", lambda: bench_multi.config4(dist, rank, world, dev, _self)),
                         ("config3", lambda: bench_multi.config3(dist, rank, world, dev, _self, c_map, 0.0155, bool(args.config3_vit))),
                         ("config5", lambda: bench_multi.config5(dist, rank, world, dev, _self))):
            try:
                multi_blocks[name] = fn()
            except Exception as ex:  # a failed block must not take the headline line with it
                multi_blocks[name] = {"error": f"{type(ex).__name__}: {ex}"[:300]}
            torch.cuda.synchronize()
            if dist is not None:
                dist.barrier()
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    peaks = measured_peaks()
    value = world * nq * args.steps / (ms / 1000.0)
    e2e_value = world * nq * args.steps / (e2e_ms / 1000.0)

    # ---- per-kernel-class times.  The timed region overlaps kernels across streams, so its event brackets include
    # cross-stream waits; the per-kernel figures (and the roofline) come from a separate pass with the overlap switched
    # off (everything on one stream: a bracket = the kernels' own time), run right after the timed region.
    _lib.check(lib.dinotrk_infer_set_overlap(0), "set_overlap")
    step_resident(); torch.cuda.synchronize()
    _lib.profile_enable(True); _lib.profile_collect()
    clean_steps = 3
    ce0, ce1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ce0.record()
    for _ in range(clean_steps):
        step_resident()
    ce1.record(); torch.cuda.synchronize()
    clean = _lib.profile_collect()
    _lib.profile_enable(False)
    _lib.check(lib.dinotrk_infer_set_overlap(-1), "set_overlap")
    serial_ms = ce0.elapsed_time(ce1) / clean_steps
    total_clean = sum(v[0] for v in clean.values()) or 1.0
    kernels = {k: {"ms_per_step": v[0] / clean_steps, "launches_per_step": v[1] / clean_steps, "share": v[0] / total_clean,
                   "ms_per_step_in_timed_region_brackets": prof.get(k, (0.0, 0))[0] / args.steps}
               for k, v in sorted(clean.items(), key=lambda kv: -kv[1][0])}
    clean_stat = {k: (v[0] * args.steps / clean_steps, v[1] * args.steps / clean_steps) for k, v in clean.items()}
    dom = max(clean.items(), key=lambda kv: kv[1][0])[0]
    roofline = kernel_roofline(dom, clean_stat[dom], args, maps_per_step, peaks, clocks, path_stats)
    extra = {k: kernel_roofline(k, clean_stat[k], args, maps_per_step, peaks, clocks, path_stats)
             for k in ("corr_gemm", "xw_coarse_gemm", "xw_exact_gemm", "xw_head", "head", "corr_stream") if k in clean_stat and k != dom}
    corr_ms = sum(clean[k][0] for k in ("corr_gemm", "xw_coarse_gemm", "xw_exact_gemm") if k in clean) / clean_steps
    if corr_ms > 0:
        ach = 2.0 * maps_per_step * P * C / (corr_ms / 1e3) / 1e12
        extra["correlation_total"] = {"kernels": [k for k in ("corr_gemm", "xw_coarse_gemm", "xw_exact_gemm") if k in clean],
                                      "bound": "tensor", "ms_per_step": corr_ms, "achieved": ach, "peak": peaks["tf_sustained"],
                                      "unit": "TFLOP/s", "frac": ach / peaks["tf_sustained"],
                                      "note": "all correlation GEMM kernels of a step together against the algorithmic 2*P*C FLOPs of "
                                              "every map (what the reference's formulation computes per map)"}
    if args.stream_probe:
        extra["corr_stream_probe"] = stream_probe(model, mi, lib, _lib, args, peaks)

    line = {"metric": "query-points/sec (854x476, T=%d)" % T, "value": value, "unit": "query-points/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(args), "T": T, "C": C, "query_points": nq,
                       "anchors_per_query_mean": n_anch.mean().item(), "corr_maps_per_step": maps_per_step,
                       "parallelism": f"video-parallel x{world}" if world > 1 else "single GPU",
                       "l2": "inputs larger than L2 (1.66 GB feature video per step; no explicit flush)",
                       "chunk_maps": args.chunk_maps, "corr_precision": args.precision, "head_kind": args.head,
                       "anchor_pipeline": path_stats["pipeline"],
                       "anchor_maps_exact_window": path_stats["exact_window"], "anchor_maps_full_map": path_stats["full_map"],
                       "anchor_maps_full_map_by_certificate": path_stats.get("full_map_by_certificate"),
                       "exact_window_fraction": (path_stats["exact_window"] / max(path_stats["anchor_maps"], 1)
                                                 if path_stats["pipeline"] == "exact-window" else None)},
            "e2e": {"value": e2e_value, "unit": "query-points/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms / args.steps},
            "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "roofline_other": extra,
            "kernels": kernels, "kernels_note": "per-class CUDA-event times of a separate overlap-off pass (%d steps, %.2f ms per "
                                                "serialised step); see the comment in bench.py" % (clean_steps, serial_ms),
            "peaks": peaks}
    for k_, v_ in multi_blocks.items():
        if v_ is not None:
            line[k_] = v_
    if args.second_head and world == 1 and args.head != "mixed":
        # the same step with mixed-sign refiner weights: whatever the head's certificate cannot cover goes through the
        # full-map refiner (a trained checkpoint's weights are not known here; this is the unfavourable end)
        model.tracker_head.load_state_dict(head_weights_for("mixed"))
        for _ in range(2):
            step_resident()
        torch.cuda.synchronize()
        st2 = _lib.infer_stats()
        m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        m0.record()
        for _ in range(3):
            step_resident()
        m1.record(); torch.cuda.synchronize()
        ms2 = m0.elapsed_time(m1) / 3
        line["second_head"] = {"head_kind": "mixed", "value": nq / (ms2 / 1e3), "unit": "query-points/s", "ms_per_step": ms2,
                               "anchor_pipeline": st2["pipeline"], "anchor_maps_exact_window": st2["exact_window"],
                               "anchor_maps_full_map": st2["full_map"]}
        model.tracker_head.load_state_dict(head_weights_for(args.head))
    if args.torch_cuda_baseline and world == 1:
        del model, mi
        torch.cuda.empty_cache()
        line["torch_cuda_baseline"] = torch_cuda_reference_sample(T, C, nq, args.noise, dev)
        line["torch_cuda_baseline"]["speedup_e2e"] = e2e_value / line["torch_cuda_baseline"]["value"]
        model = mi = None
    if args.stages and world == 1:
        line["stages"] = stage_timings(args, dev, _lib, peaks)
        line["stages"]["train_step"] = train_step_stage(args, dev, _lib, bool(args.torch_cuda_baseline))
        fs = line["stages"]["per_video_feature_stage_s"]
        line["stages"]["query_points_per_s_from_pixels"] = nq / (fs + ms / args.steps / 1000.0)
    if args.cpu_baseline and world == 1:
        v, cores, desc, _, spread = cpu_reference_sample(T, C, nq, args.noise, seed=0, anchor_calls=3, samples=3)
        line["cpu_baseline"] = {"value": v, "unit": "query-points/s", "cores": cores, "kind": "port", "sample": desc,
                                "spread": spread}
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def ncu_traffic(csv_name):
    """dram__bytes_read.sum + dram__bytes_write.sum of the committed `ncu --set full` capture (profiles/), bytes per launch."""
    path = os.path.join(ROOT, "profiles", csv_name)
    if not os.path.exists(path):
        return None
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    tot, seen = 0.0, 0
    for line in open(path):
        f = line.strip().split(",")
        if f[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum") and len(f) >= 3:
            tot += float(f[2].strip('"')) * unit.get(f[1], 1.0)
            seen += 1
    return tot if seen == 2 else None


def kernel_roofline(name, stat, args, maps_per_step, peaks, clocks, path_stats=None):
    """Algorithmic work per launch / average launch time for one kernel class (DESIGN.md section 4 states the per-unit figures)."""
    ms_total, launches = stat
    avg_s = ms_total / 1000.0 / max(launches, 1)
    anchor_maps = (path_stats or {}).get("anchor_maps", 0)
    xw = (path_stats or {}).get("pipeline") == "exact-window"
    # maps a launch of this class processes: the exact-window kernels only see the anchor phase
    if name.startswith("xw_"):
        maps_total = anchor_maps * args.steps
    elif name in ("corr_gemm", "head", "head_full") and xw:
        maps_total = (maps_per_step - anchor_maps + (path_stats or {}).get("full_map", 0)) * args.steps
    else:
        maps_total = maps_per_step * args.steps
    maps_per_launch = maps_total / max(launches, 1)
    tensor_note = "peak = sustained cuBLAS bf16 (%s)" % peaks["which"]
    if name == "xw_coarse_gemm":
        flops = 2.0 * maps_per_launch * P * args.C
        ach = flops / avg_s / 1e12
        return {"kernel": name, "bound": "tensor", "achieved": ach, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                "frac": ach / peaks["tf_sustained"], "traffic": ncu_traffic("ncu_r2_xw_coarse.csv"),
                "traffic_note": "DRAM read + write bytes per launch from the committed ncu --set full capture of this kernel "
                                "(profiles/ncu_r2_xw_coarse.csv), null until captured; algorithmic bytes per map: fp16 operands "
                                "(descriptor 2 KB + its share of the frame's 16.6 MB) + 384 B of tile keys -- no map is stored",
                "note": "single kind::f16 pass over the hi halves: executed MMA FLOPs = algorithmic 2*maps*P*C; " + tensor_note,
                "maps_per_launch": maps_per_launch, "ms_per_launch": avg_s * 1e3}
    if name == "xw_exact_gemm":
        cell = max(args.T if args.T <= 128 else 125, 1)                 # maps per cell; UMMA N = 64 or 128 columns
        flops_exec = 2.0 * maps_per_launch * 512 * args.C * 3 * ((64.0 if cell <= 64 else 128.0) / cell)
        flops_alg = 2.0 * maps_per_launch * 225 * args.C
        ach = flops_alg / avg_s / 1e12
        return {"kernel": name, "bound": "tensor", "achieved": ach, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                "frac": ach / peaks["tf_sustained"], "traffic": ncu_traffic("ncu_r2_final_xw.csv"),
                "executed_mma_tflops": flops_exec / avg_s / 1e12,
                "note": "algorithmic = the 15 x 15 window the head needs per map (2*225*C FLOPs); executed = 3 split-precision "
                        "passes x 512 box-token rows (4 parts of 128, 441 used) x 64 UMMA columns per cell of T <= 64 maps; "
                        "traffic: profiles/ncu_r2_final_xw.csv, first kernel; " + tensor_note,
                "maps_per_launch": maps_per_launch, "ms_per_launch": avg_s * 1e3}
    if name in ("corr_gemm", "best_buddies", "vit_gemm", "delta_conv"):
        flops = 2.0 * maps_per_launch * P * args.C  # <d, F[p]> for every token of the target frame
        ach = flops / avg_s / 1e12
        return {"kernel": name, "bound": "tensor", "achieved": ach, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                "frac": ach / peaks["tf_sustained"],
                "traffic": None,
                "note": ("algorithmic FLOPs = 2*maps*P*C per launch; %s. precision=%s: "
                         "fp16x3 executes 3 kind::f16 MMA passes (lo*hi, hi*lo, hi*hi) per algorithmic FLOP, so the tensor "
                         "pipe is busy ~3x this fraction; fp32 = exact FFMA GEMM on the CUDA cores") % (tensor_note, args.precision),
                "executed_mma_tflops": ach * 3 if args.precision == "fp16x3" else None,
                "maps_per_launch": maps_per_launch, "ms_per_launch": avg_s * 1e3}
    if name in ("head", "xw_head"):
        # the windowed refiner: 169*16*9 + 121*16*9 = 41 760 FMA per map
        # (the reference's full-map formulation, SURVEY.md 8a row a7, is 4.67 MFLOP per map: 56x more)
        flops = 2.0 * 41760 * maps_per_launch
        ach = flops / avg_s / 1e12
        pk = fp32_peak_tflops(clocks)
        return {"kernel": name, "bound": "fp32-cuda-core", "achieved": ach, "peak": pk, "unit": "TFLOP/s",
                "frac": ach / pk, "traffic": None, "ns_per_map": avg_s * 1e9 / max(maps_per_launch, 1),
                "reference_formulation_tflops": 4.67e6 * maps_per_launch / avg_s / 1e12,
                "note": ("exact-fp32 CUDA-core work of the windowed refiner (83.5 kFLOP per map; the full-map formulation the "
                         "reference evaluates is 4.67 MFLOP per map and is only run for uncertified maps); "
                         "peak = 148 SMs x 128 lanes x 2 x max SM clock")}
    return {"kernel": name, "bound": "hbm", "achieved": None, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": None,
            "traffic": None, "note": "see roofline_other.corr_stream_probe"}


def stage_timings(args, dev, _lib, peaks, vit_only=False):
    """Per-video preprocessing stages on real shapes (854x476): ViT feature extraction (a1), delta-DINO refinement
    (a2) and best-buddies (a13), device-timed.  Random-init weights of the named architectures."""
    from dino_tracker_b200.vit import DinoV2Features, CONFIGS
    from dino_tracker_b200.networks import DeltaDINO
    from dino_tracker_b200.best_buddies import nearest_neighbours
    out = {}
    name = "dinov2_vitl14" if args.C == 1024 else "dinov2_vitb14"
    depth, dim, heads = CONFIGS[name]
    layer = 15 if args.C == 1024 else depth - 1
    g = torch.Generator(device=dev).manual_seed(7)

    def rn(*shape, std=0.02):
        return torch.randn(*shape, device=dev, generator=g) * std
    sd = {"cls_token": rn(1, 1, dim), "pos_embed": rn(1, 1 + 37 * 37, dim), "patch_embed.proj.weight": rn(dim, 3, 14, 14),
          "patch_embed.proj.bias": rn(dim)}
    for i in range(layer + 1):
        p = f"blocks.{i}."
        sd.update({p + "norm1.weight": 1 + rn(dim), p + "norm1.bias": rn(dim), p + "attn.qkv.weight": rn(3 * dim, dim),
                   p + "attn.qkv.bias": rn(3 * dim), p + "attn.proj.weight": rn(dim, dim), p + "attn.proj.bias": rn(dim),
                   p + "ls1.gamma": 1 + rn(dim), p + "norm2.weight": 1 + rn(dim), p + "norm2.bias": rn(dim),
                   p + "mlp.fc1.weight": rn(4 * dim, dim), p + "mlp.fc1.bias": rn(4 * dim),
                   p + "mlp.fc2.weight": rn(dim, 4 * dim), p + "mlp.fc2.bias": rn(dim), p + "ls2.gamma": 1 + rn(dim)})
    ex = DinoV2Features(sd, heads=heads, layer=layer, device=dev, frames_per_call=2)
    frames = torch.rand(2, 3, H, W, device=dev, generator=g)

    def timed(fn, reps):
        fn(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        _lib.profile_enable(True); _lib.profile_collect()
        e0.record()
        for _ in range(reps):
            fn()
        e1.record(); torch.cuda.synchronize()
        prof = _lib.profile_collect(); _lib.profile_enable(False)
        return e0.elapsed_time(e1) / reps, {k: round(v[0] / reps, 3) for k, v in prof.items()}

    ms, prof = timed(lambda: ex(frames), 2)
    flops = 2.0 * (12 * dim * dim * (P + 1) + 2 * (P + 1) ** 2 * dim) * (layer + 1) * frames.shape[0]
    out["vit"] = {"model": f"{name}@block{layer}", "frames_per_s": frames.shape[0] / (ms / 1000), "ms_per_frame": ms / frames.shape[0],
                  "tflops": flops / (ms / 1000) / 1e12, "frac_of_bf16_peak": flops / (ms / 1000) / 1e12 / peaks["tf_sustained"],
                  "kernel_ms_per_call": prof, "math": "kind::f16 tcgen05 GEMMs (fp16 operands, fp32 accumulate, fp32 residual stream) + fused tcgen05 attention"}
    del ex, sd
    if vit_only:
        return out
    # delta-DINO with the shipped channel widths
    dd = DeltaDINO(channels=[3, 64, 128, 256, args.C]).to(dev)
    torch.nn.init.normal_(dd.layers[12].weight, std=0.01)
    geom = _lib.make_geom(H, W)
    dino = torch.randn(4, P, args.C, device=dev, generator=g)
    fr4 = torch.rand(4, 3, H, W, device=dev, generator=g)
    ms, prof = timed(lambda: dd.refine_tpc(fr4, dino, geom), 2)
    out["delta_dino"] = {"frames_per_s": 4 / (ms / 1000), "ms_per_frame": ms / 4, "tflops": 171.4e9 * 4 / (ms / 1000) / 1e12,
                         "kernel_ms_per_call": prof,
                         "math": "convs = im2col (fp16 hi/lo split) + tcgen05 split-precision GEMMs, fp32-faithful"}
    del dd
    # pixels -> tracks for one video of the bench shape: ViT + delta-DINO once per video, then the tracker step
    per_video_s = (out["vit"]["ms_per_frame"] + out["delta_dino"]["ms_per_frame"]) * args.T / 1000.0
    out["per_video_feature_stage_s"] = per_video_s
    # best buddies: 4 frames -> 12 ordered pairs
    feats = dino
    norms = feats.norm(dim=2).contiguous()
    pairs = [(s, t) for s in range(4) for t in range(4) if s != t]
    ms, prof = timed(lambda: nearest_neighbours(feats, norms, geom, pairs), 2)
    out["best_buddies"] = {"ordered_pairs_per_s": len(pairs) / (ms / 1000), "ms_per_ordered_pair": ms / len(pairs),
                           "tflops": 2.0 * P * P * args.C * len(pairs) / (ms / 1000) / 1e12, "kernel_ms_per_call": prof,
                           "math": "tcgen05 3xTF32 GEMM + top-2 epilogue + exact fp32 resolve"}
    return out


def train_step_stage(args, dev, _lib, torch_baseline):
    """The tracker node of one training iteration (dino_tracker.py:405-411) at the reference's batch shape
    (config/train.yaml: train_batch_size 512 points, batch_n_frames 4): forward with the graph and the CUDA reverse
    pass down to d loss / d embeddings and d loss / d refiner weights, device-timed; beside it (optional) the same node
    as PyTorch-CUDA autograd through the oracle's restatement (exact fp32) -- what the reference's trainer executes."""
    from dino_tracker_b200 import Tracker
    N, B = 4, 512
    feats = synth_video_features(N, args.C, dev, seed=3, noise=args.noise)
    head = head_weights_for(args.head)
    m = Tracker(video=torch.zeros(N, 3, H, W, device=dev), dino_embed_video=feats, device=dev, delta_channels=[3, 8, 8, 8, args.C])
    m.tracker_head.load_state_dict(head)
    cg = torch.Generator().manual_seed(12)
    pts = (torch.rand(B, 3, generator=cg) * torch.tensor([W - 1.0, H - 1.0, 0.0])).to(dev)
    src = torch.randint(0, N, (B,), generator=cg).to(dev)
    tgt = torch.randint(0, N, (B,), generator=cg).to(dev)
    labels = (torch.rand(B, 2, generator=cg) * 2 - 1).to(dev)
    fs = torch.arange(N, dtype=torch.int32, device=dev)
    huber = torch.nn.HuberLoss(delta=1 / 32, reduction="none")

    def run(forward, reps):
        f_ms, b_ms = [], []
        for i in range(reps + 1):
            e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            e[0].record()
            loss = huber(forward(), labels).mean()
            e[1].record()
            loss.backward()
            e[2].record(); torch.cuda.synchronize()
            if i:       # first pass = warm-up
                f_ms.append(e[0].elapsed_time(e[1])); b_ms.append(e[1].elapsed_time(e[2]))
        return sum(f_ms) / reps, sum(b_ms) / reps

    emb = feats.clone().requires_grad_(True)
    _lib.profile_enable(True); _lib.profile_collect()
    f_ms, b_ms = run(lambda: m.get_point_predictions((pts, src, tgt, fs), emb), 3)
    prof = _lib.profile_collect(); _lib.profile_enable(False)
    out = {"batch_points": B, "frames": N, "C": args.C, "forward_ms": f_ms, "backward_ms": b_ms,
           "kernel_ms_per_step": {k: round(v[0] / 4, 3) for k, v in prof.items()},
           "gradients": "embeddings [4][8107][C] + normalised refiner weights (305)",
           "note": "tracker node only; delta-DINO's convolutions / BatchNorm of the training graph are torch (cuDNN) ops"}
    if torch_baseline:
        import oracle
        from oracle import tracker as ot
        oracle.use_exact_fp32()
        geo = ot.Geometry(H=H, W=W)
        f_o = feats.clone().requires_grad_(True)
        head_o = {k: v.to(dev).requires_grad_(True) for k, v in head.items()}
        tf_ms, tb_ms = run(lambda: ot.tracker_forward(f_o, (pts, src, tgt, fs), head_o, geo), 2)
        out["torch_cuda_autograd"] = {"forward_ms": tf_ms, "backward_ms": tb_ms,
                                      "speedup": (tf_ms + tb_ms) / (f_ms + b_ms)}
    return out


def fp32_peak_tflops(clocks):
    mhz = (clocks or {}).get("sm_max_mhz") or 1965.0
    return 148 * 128 * 2 * mhz * 1e6 / 1e12


def stream_probe(model, mi, lib, _lib, args, peaks):
    """The HBM-bound correlation kernel of SURVEY.md 8d on its own: Q_b descriptors x all T frames in one
    launch (trajectory phase of a small query batch).  Algorithmic bytes per pass =
    T*P*C*4 + T*P*4 + Q_b*C*4 + Q_b*T*8."""
    import ctypes
    dev = model._dev
    T, C = args.T, args.C
    out = {}
    for qb in (1, 8, 9, 32, 128, 256):
        # one descriptor row per map (the entry point's contract): the Q_b descriptors repeated for every frame
        desc = torch.randn(qb, C, device=dev).repeat(T, 1).contiguous()
        dn = desc.norm(dim=1).contiguous()
        grp = torch.stack([torch.arange(T), torch.arange(T) * qb, torch.full((T,), qb),
                           torch.arange(T) * qb]).to(torch.int32).to(dev).contiguous()
        stride = lib.dinotrk_map_stride(ctypes.byref(model._geom))
        maps = torch.empty(T * qb, stride, device=dev)
        nb = lib.dinotrk_corr_maps_workspace_bytes(T * qb, T, C)
        ws = torch.empty(nb, device=dev, dtype=torch.uint8)
        feat = model.features_struct(model._refined_tpc, model._refined_norms)

        def run():
            _lib.check(lib.dinotrk_corr_maps(ctypes.byref(feat), ctypes.byref(model._geom), _lib.ptr(desc), _lib.ptr(dn),
                                             _lib.ptr(grp[0]), _lib.ptr(grp[1]), _lib.ptr(grp[2]), _lib.ptr(grp[3]), T,
                                             T * qb, qb, _lib.ptr(maps), _lib.ptr(ws), nb, _lib.stream_ptr()))
        for _ in range(3):
            run()
        torch.cuda.synchronize()
        _lib.profile_enable(True); _lib.profile_collect()
        for _ in range(5):
            run()
        prof = _lib.profile_collect(); _lib.profile_enable(False)
        if qb <= 8:                    # <= 8 descriptors per frame: the HBM-bound streaming kernel (exact fp32)
            ms_total, n = prof["corr_stream"]
            nbytes = T * P * C * 4 + T * P * 4 + qb * C * 4 + qb * T * 8
            gbs = nbytes / (ms_total / n / 1000.0) / 1e9
            out[f"Q_b={qb}"] = {"kernel": "corr_stream", "bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"],
                                "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"], "traffic": None,
                                "bytes_per_launch": nbytes, "ms_per_launch": ms_total / n}
        else:                          # wider groups: split-precision tensor GEMM (128-row tiles up to 128 descriptors)
            ms_total, n = prof["corr_gemm"]
            fl = 2.0 * qb * T * P * C
            tf = fl / (ms_total / n / 1000.0) / 1e12
            out[f"Q_b={qb}"] = {"kernel": "corr_gemm (full maps, 3 fp16 passes)", "bound": "tensor", "achieved": tf,
                                "peak": peaks["tf_sustained"], "unit": "TFLOP/s", "frac": tf / peaks["tf_sustained"],
                                "traffic": None, "ms_per_launch": ms_total / n,
                                "tile_rows": 128 if qb <= 128 else 256}
    return out


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
