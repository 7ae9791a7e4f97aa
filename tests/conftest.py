import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def mnist_golden():
    """The reference's bundled MNIST fixtures; ``content_holo`` [20,5,K] holds each hologram at the flat positions
    ``holo_idx`` of its 128 x 128 image (oracle/make_golden.py)."""
    from oracle import make_golden
    g = dict(np.load(os.path.join(GOLDEN, "mnist_holo.npz")))
    g["gt_phase"] = make_golden.PHASE_LEVELS[g.pop("gt_phase_code")]
    return g


@pytest.fixture(scope="session")
def ref_cases():
    """The reference's outputs (image-sized ones at the positions ``<case>.idx``, see make_golden.at) together with the
    inputs they were computed from, drawn again from the seeded generator and checked against the stored CRCs."""
    from oracle import make_golden
    c = dict(np.load(os.path.join(GOLDEN, "ref_cases.npz")))
    for k, v in make_golden.ref_case_inputs().items():
        name, key = k.split(".", 1)
        if key != "meta":
            assert make_golden.crc(v) == c[f"{name}.crc.{key}"], f"{k} no longer regenerates from the stored seed"
        c[k] = v
    return c
