"""The committed fixtures against a separate record of what the UNMODIFIED reference computes on a few small seeded inputs
(tests/golden/reference_live.npz, written by `python tests/golden/make_golden.py --only live`, which runs the reference
through oracle/refshim.py), so the goldens are demonstrably what the reference produces -- not a stale copy."""
import hashlib
import json

import numpy as np

from conftest import golden_path


def test_fixtures_are_live_reference_outputs():
    out = np.load(golden_path("reference_live.npz"))
    gold = json.load(open(golden_path("path_index.json")))
    assert str(out["path_sha"]) == gold["r5_21x26"]["sha256"]
    g = np.load(golden_path("affinity_12x17.npz"))
    assert str(out["aff_sha"]) == hashlib.sha256(np.ascontiguousarray(g["aff"]).tobytes()).hexdigest()
    g = np.load(golden_path("rw_%s.npz" % out["rw_name"]))
    t = np.load(golden_path("to_affinity.npz"))
    assert str(out["toaff_sha"]) == hashlib.sha256(np.ascontiguousarray(t["r5_aff"]).tobytes()).hexdigest()
    assert np.abs(out["toaff_grad"].reshape(t["r5_grad_edge"].shape) - t["r5_grad_edge"]).max() < 1e-5
    live = out["rw"].reshape(g["rw"].shape)
    # same code, same seeds, same machine class: the matrix products may differ in the last bits between BLAS builds / thread counts
    assert np.abs(live - g["rw"]).max() < 1e-6
