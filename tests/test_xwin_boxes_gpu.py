"""GPU: the exact-window pipeline's per-cell token boxes (csrc/xwin.cu) on a 'plateau' feature video.

The box of a cell is fitted to the arg-max candidates of its fitting members: 16 columns x 2..3 parts of 8 rows when they
span <= 2 columns, else 21 columns x 3..4 parts of 6 rows.  Translating fields with sharp correlation peaks put nearly every
cell in a 2-part box; here the field is smoothed many times, so the peaks are flat and the members of a cell disagree by
a few tokens -- the call sees several box shapes, which must all agree with the full-map pipeline and the oracle."""
import numpy as np
import pytest
import torch

from oracle import inference as oi
from oracle import synth
from oracle.tracker import Geometry
from test_xwin_gpu import XY_TOL, _agree, _run

pytestmark = pytest.mark.gpu


def plateau_features(T, C, h, w, seed, noise, max_shift, passes):
    """synth.shifted_field_features with `passes` smoothing passes and the field rescaled to unit standard deviation
    before the per-frame noise is added."""
    rs = np.random.RandomState(seed)
    pad = max_shift * 2 + 2
    base = rs.standard_normal((C, h + 2 * pad, w + 2 * pad)).astype(np.float32)
    for _ in range(passes):
        b = base.copy()
        b[:, 1:-1, 1:-1] = (base[:, 1:-1, 1:-1] * 0.5 + 0.125 * (base[:, :-2, 1:-1] + base[:, 2:, 1:-1]
                            + base[:, 1:-1, :-2] + base[:, 1:-1, 2:]))
        base = b
    base /= base.std()
    shifts = np.zeros((T, 2), dtype=np.int64)
    for t in range(1, T):
        shifts[t] = np.clip(shifts[t - 1] + rs.randint(-1, 2, size=2), -max_shift, max_shift)
    feats = np.empty((T, C, h, w), dtype=np.float32)
    for t in range(T):
        dy, dx = shifts[t]
        feats[t] = base[:, pad + dy: pad + dy + h, pad + dx: pad + dx + w]
        feats[t] += noise * rs.standard_normal((C, h, w)).astype(np.float32)
    return torch.from_numpy(feats)


def test_plateau_cells_take_several_box_shapes():
    geo = Geometry()
    T, C = 6, 128
    feats = plateau_features(T, C, geo.h, geo.w, seed=21, noise=1.0, max_shift=2, passes=16)
    head = synth.head_weights("sharp", seed=T)
    q = synth.lattice_query_points(5, 4, geo.H, geo.W, t_q=[i % T for i in range(20)], margin=30.0, jitter_seed=T)
    full, _ = _run(feats, head, q, geo, 0)
    xw, st = _run(feats, head, q, geo, 1)
    assert st["pipeline"] == "exact-window"
    d = _agree(xw, full)
    parts = st["exact_window_cells_by_parts"]
    print(f"plateau: exact-window vs full-map max |dxy| = {d:.2e} px; {st}")
    assert st["exact_window"] + st["full_map"] == st["anchor_maps"] == int((xw["cos_sims"] >= 0.7).sum().item()) * T
    assert st["exact_window"] >= 0.5 * st["anchor_maps"]
    assert sum(1 for v in parts.values() if v > 0) >= 2, parts       # several box shapes in one call
    assert parts[4] > 0, parts                                       # 4 parts: only a 21-wide box has them
    t_ref, o_ref, aux = oi.infer(feats, q, head, geo, 0.7, 0.6, return_all=True)
    assert (xw["traj"].cpu() - aux["trajs"]).abs().max().item() <= XY_TOL
    assert torch.equal(xw["occ"].bool().cpu(), o_ref)
    vis = aux["cos_sims"] >= 0.7
    for n in range(q.shape[0]):
        assert (xw["anchors"][n].cpu()[vis[n]] - aux["anchors"][n]).abs().max().item() <= XY_TOL
