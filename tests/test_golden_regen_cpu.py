"""The training-step and cycle-consistency fixtures are, bit for bit, what the reference returned, and the seeded
generators still produce, bit for bit, the inputs it was given.  Both are pinned by tests/golden/reference_digests.json,
recorded from a run of the reference (`python -m oracle.make_golden` rewrites every fixture and the digests)."""
import json
import os

import numpy as np
import pytest

from oracle import make_golden as mg

from golden_util import GOLDEN_DIR

DIGESTS = json.load(open(os.path.join(GOLDEN_DIR, "reference_digests.json")))


@pytest.mark.parametrize("name,inputs", [("train_small", "train_case_arrays"), ("cycle_small", "cycle_case_arrays")])
def test_fixture_matches_the_recorded_reference_run(name, inputs):
    want = DIGESTS[name]
    got = {k: mg.array_digest(v) for k, v in getattr(mg, inputs)().items()}
    assert got == want["inputs"], sorted(k for k in set(got) | set(want["inputs"]) if got.get(k) != want["inputs"].get(k))
    fixture = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    got = {k: mg.array_digest(fixture[k]) for k in fixture.files}
    assert got == want["outputs"], sorted(k for k in set(got) | set(want["outputs"]) if got.get(k) != want["outputs"].get(k))
