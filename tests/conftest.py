import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


class _Fixture(dict):
    """A fixture with arrays added after loading; ``files`` lists its keys like ``NpzFile.files``."""

    @property
    def files(self):
        return list(self)


def load_golden(name):
    g = np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False)
    if "uvs_sha256" not in g.files:
        return g
    # Observations too large to store (ba_cfg1: 1.7 MB of noise) are kept as the scene generator's
    # arguments and the SHA-256 of the array the reference ran on; the regenerated array must match it
    # bit for bit, so a drifted generator fails here instead of testing against other inputs.
    import hashlib
    import json
    from multicam_calibration_b200.synthetic import make_scene
    d = _Fixture((k, g[k]) for k in g.files)
    uvs = np.ascontiguousarray(make_scene(**json.loads(str(d["scene"]))).uvs, dtype=np.float64)
    assert hashlib.sha256(uvs.tobytes()).hexdigest() == str(d["uvs_sha256"]), \
        f"{name}.npz: the scene generator no longer reproduces the observations of the fixture"
    d["uvs"] = uvs
    return d


@pytest.fixture(scope="session")
def golden():
    return load_golden


def split_cams(cams):
    """(C,12) camera rows -> (extrinsics (C,6), intrinsics list) in the reference's types."""
    intr = []
    for p in cams:
        K = np.eye(3)
        K[0, 0], K[1, 1], K[0, 2], K[1, 2] = p[:4]
        intr.append((K, np.r_[p[4:6], 0.0, 0.0, 0.0]))
    return cams[:, 6:].copy(), intr
