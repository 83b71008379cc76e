import glob
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def golden_files(prefix):
    return sorted(glob.glob(os.path.join(GOLDEN, prefix + "_*.npz")))


def load_golden(path):
    with np.load(path) as z:
        return {k: z[k] for k in z.files}

