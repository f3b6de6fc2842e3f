"""Bit-identity of the bench workload's outputs across kernel optimisations.

The C2 configuration (Zig-Zag, banana potential, d = 50, Brent constant bounds, Philox draws) runs on the team-of-8
transposed Brent kernel at a reduced size, and every history array and the closed-form segment moments are hashed
byte for byte.  A Boomerang run covers the rotation-flow branch of the moment kernel.  The digests in
golden/c2_identity_sha256.json were written by the build before the team kernel's batched rate evaluation and the
streaming moment kernel; these changes only reorder independent work or skip additions of exactly +0.0, so the
outputs must not move by a single bit.

Regenerate (only when a change is meant to alter results): python tests/test_gpu_c2_identity.py --write
"""
import hashlib
import json
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
DIGESTS = os.path.join(HERE, "golden", "c2_identity_sha256.json")
HISTORY_FIELDS = ("X", "V", "t", "horizon", "ar", "error_value_ar", "errored_bound", "rejected", "hitting_horizon",
                  "tape_pos", "counters", "status")


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _run(p, sampler, x0, v0, n_sk, seed, team):
    if team:
        os.environ["PDMPFLUX_TEAM"] = str(team)
    try:
        h = p.sample_skeleton(sampler, n_sk, x0, v0, seed=seed)
    finally:
        os.environ.pop("PDMPFLUX_TEAM", None)
    m1, m2, T = p.skeleton_moments(sampler, h)
    out = {f: _sha(getattr(h, f)) for f in HISTORY_FIELDS}
    out.update(m1=_sha(m1), m2=_sha(m2), T=_sha(T))
    return out


def compute_digests():
    if os.path.dirname(HERE) not in sys.path:
        sys.path.insert(0, os.path.dirname(HERE))
    import pdmpflux_b200 as p

    g = np.random.default_rng(20261020)
    nch, n_sk, d = 512, 200, 50
    x0 = g.standard_normal((nch, d))
    v0 = np.where(g.random((nch, d)) < 0.5, -1.0, 1.0)
    res = {"c2_team8": _run(p, p.ZigZag(d, p.Banana(), grid_size=0), x0, v0, n_sk, 2024, 8)}
    nb, nbs, db = 256, 200, 20
    xb = g.standard_normal((nb, db)); vb = g.standard_normal((nb, db))
    res["boomerang_gauss20"] = _run(p, p.Boomerang(db, p.GaussStd()), xb, vb, nbs, 7, None)
    return res


@pytest.mark.gpu
def test_c2_outputs_bit_identical():
    with open(DIGESTS) as f:
        want = json.load(f)
    got = compute_digests()
    for case, arrays in want.items():
        for name, digest in arrays.items():
            assert got[case][name] == digest, f"{case}: {name} differs from the recorded build"


if __name__ == "__main__":
    if "--write" in sys.argv:
        with open(DIGESTS, "w") as f:
            json.dump(compute_digests(), f, indent=1, sort_keys=True)
            f.write("\n")
    else:
        print(json.dumps(compute_digests(), indent=1, sort_keys=True))
